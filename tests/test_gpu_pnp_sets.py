"""The all / full-mask / visible-mask poses of every RoI in one PnP launch (cp_pnp_ransac_sets, ops.pnp_ransac with a tuple
``flag``, forward_with_pose with a tuple ``flag``).

Contract: slab v of a launch over the flag masks (m_0, ..., m_{V-1}) equals, bit for bit, cp_pnp_ransac with flag_mask = m_v
and the same seed, graph_sel, cam_K and iteration count; with ``rng_index`` RoI b equals row rng_index[b] of the launch over
the batch that index refers to.  The scenes are those of tests/test_gpu_pnp.py (shipped FPS clouds under random poses, the
LM camera, 20 % outliers, 10 % of the keypoints outside the RoI), with per-RoI full and visible masks cut out of the grid."""
import numpy as np
import pytest
import torch

from helpers import syn
from test_gpu_pnp import K_LM, TOL_R_DEG, TOL_T_MM, cv2_pose, rot_err_deg, scene

pytestmark = pytest.mark.gpu

ALL, FULL, VISIB = 1, 2, 4
FLAG_TUPLES = [(1, 2, 4), (4, 2, 1), (2, 4), (4, 1), (1,), (4,), (3, 6, 5)]
SEED = 11


@pytest.fixture(scope="module")
def ops():
    from checkerpose_b200 import ops as o
    return o


def _masks(scenes, seed, degenerate=True):
    """(B, 2, 64, 64) seg logits: channel 1 (full mask) drops a band of rows, channel 0 (visible mask) also drops a band of
    columns (an occluder).  With ``degenerate``, every 7th RoI (from 3) has an empty full mask and every 7th (from 5) keeps
    only the cells of 3 keypoints that have a cell to themselves in its visible mask: fewer than 4 entries in that set only."""
    rng = np.random.default_rng(seed)
    B = len(scenes)
    seg = np.full((B, 2, 64, 64), 2.0, dtype=np.float32)
    for b, s in enumerate(scenes):
        r, c = int(rng.integers(0, 12)), int(rng.integers(0, 20))
        seg[b, :, :r, :] = -2.0
        side = rng.random() < 0.5
        if side:
            seg[b, 0, :, :c] = -2.0
        else:
            seg[b, 0, :, 64 - c:] = -2.0
        if degenerate and b % 7 == 3:
            seg[b, 1] = -2.0
        if degenerate and b % 7 == 5:
            xid, yid, roi = s[4], s[5], s[6] > 0
            cells = yid * 64 + xid
            cnt = np.bincount(cells[roi], minlength=64 * 64)
            lone = [k for k in np.flatnonzero(roi) if cnt[cells[k]] == 1][:3]
            seg[b, 0] = -2.0
            for k in lone:
                seg[b, 0, yid[k], xid[k]] = 2.0
    return seg


def _batch(ops, ds, objs, N, B, seed, degenerate=True, scenes=None):
    """B RoIs cycling over ``objs`` -> (scenes, packed rows, 12-byte records, clouds (G,N,3), per-RoI cloud index)."""
    scenes = scenes or [scene(ds, objs[b % len(objs)], N, seed + 13 * b) for b in range(B)]
    roi = torch.tensor(np.stack([s[6] for s in scenes])).view(B, 1, N).cuda()
    seg = torch.from_numpy(_masks(scenes, seed, degenerate)).cuda()
    bbox = torch.tensor(np.stack([s[3] for s in scenes])).cuda()
    xid = torch.tensor(np.stack([s[4] for s in scenes])).cuda()
    yid = torch.tensor(np.stack([s[5] for s in scenes])).cuda()
    packed = ops.correspondences_packed(roi, seg, bbox, xid, yid)
    rec = ops.correspondences(roi, seg, bbox, xid, yid)
    clouds = torch.tensor(np.stack([syn.load_fps_xyz(ds, o, N) for o in objs]), dtype=torch.float32).cuda()
    sel = torch.tensor([b % len(objs) for b in range(B)], dtype=torch.int32).cuda()
    return scenes, packed, rec, clouds, sel


def _cams(B, seed):
    """Per-RoI intrinsics: the LM camera with the focal lengths and principal point jittered by a few pixels."""
    g = torch.Generator().manual_seed(seed)
    K = torch.tensor(K_LM, dtype=torch.float32).repeat(B, 1, 1)
    K[:, 0, 0] += torch.rand(B, generator=g) * 8 - 4
    K[:, 1, 1] += torch.rand(B, generator=g) * 8 - 4
    K[:, :2, 2] += torch.rand(B, 2, generator=g) * 6 - 3
    return K.cuda()


def _set_sizes(ops, packed, masks):
    _, flags, _, _, _ = ops.unpack_correspondences_host(packed)
    return {m: ((flags & m) != 0).sum(1) for m in masks}


def _check_sets_equal_single(ops, records, clouds, K, sel, flags, **kw):
    R, t, n, m = ops.pnp_ransac(records, clouds, K, graph_sel=sel, flag=flags, seed=SEED, return_inlier_mask=True, **kw)
    V, B = len(flags), records.shape[0]
    assert R.shape == (V, B, 3, 3) and t.shape == (V, B, 3) and n.shape == (V, B) and m.shape[:2] == (V, B)
    for v, f in enumerate(flags):
        R1, t1, n1, m1 = ops.pnp_ransac(records, clouds, K, graph_sel=sel, flag=f, seed=SEED, return_inlier_mask=True)
        assert torch.equal(R[v], R1) and torch.equal(t[v], t1), f"pose of set {v} (flag {f}) of {flags}"
        assert torch.equal(n[v], n1) and torch.equal(m[v], m1), f"inliers of set {v} (flag {f}) of {flags}"
    return R, t, n


# N, B, dataset, objects: B ragged, and more than one wave of 148 CTAs per set
KERNEL_CASES = [(512, 151, "lmo", (1, 5, 6, 8, 9)), (1024, 37, "lm", (3, 9, 11)), (4096, 300, "ycbv", (2, 5, 15, 21))]


@pytest.mark.parametrize("N, B, ds, objs", KERNEL_CASES)
@pytest.mark.parametrize("records", ["packed", "rec12"])
@pytest.mark.parametrize("clouds", ["shared", "graph_sel"])
@pytest.mark.parametrize("cam", ["shared", "batched"])
def test_sets_equal_single_flag_launches(ops, N, B, ds, objs, records, clouds, cam):
    scenes, packed, rec, P, sel = _batch(ops, ds, objs if clouds == "graph_sel" else objs[:1], N, B, 1000 + N)
    if clouds == "shared":
        P, sel = P[:1], None
    K = _cams(B, N) if cam == "batched" else torch.tensor(K_LM, dtype=torch.float32).cuda()
    inp = packed if records == "packed" else rec
    sizes = _set_sizes(ops, packed, (ALL, FULL, VISIB))
    degenerate = [b for b in range(B) if sizes[FULL][b] < 4 or sizes[VISIB][b] < 4]
    assert len(degenerate) >= 2 * (B // 7) and all(sizes[ALL][b] >= 4 for b in degenerate)
    for flags in FLAG_TUPLES:
        R, t, n = _check_sets_equal_single(ops, inp, P, K, sel, flags)
        for v, f in enumerate(flags):
            few = torch.from_numpy(_set_sizes(ops, packed, (f,))[f] < 4).cuda()
            assert few.sum() > 0 or f not in (FULL, VISIB)
            assert torch.equal(R[v][few], torch.eye(3, device="cuda").expand(int(few.sum()), 3, 3))
            assert float(t[v][few].abs().sum()) == 0.0 and int(n[v][few].abs().sum()) == 0
            if cam == "shared":       # the camera the scenes were projected with: every set of 4 or more entries has a pose
                assert bool((n[v][~few] > 0).all()), f"flag {f}: a set with 4 or more entries found no pose"


@pytest.mark.parametrize("cam", ["shared", "batched"])
def test_rng_index_draws_the_full_batch_hypotheses(ops, cam):
    """A permuted sub-batch launched with rng_index = the RoIs' indices in the full batch equals those rows of the full-batch
    launch, for one flag and for three."""
    N, B = 1024, 160
    _, packed, _, P, sel = _batch(ops, "ycbv", (4, 7, 12), N, B, 77)
    K = _cams(B, 3) if cam == "batched" else torch.tensor(K_LM, dtype=torch.float32).cuda()
    idx = torch.randperm(B, generator=torch.Generator().manual_seed(5))[:97].cuda()
    Ks = K[idx] if cam == "batched" else K
    for flags in ((ALL, FULL, VISIB), (VISIB, ALL), FULL):
        full = ops.pnp_ransac(packed, P, K, graph_sel=sel, flag=flags, seed=SEED, return_inlier_mask=True)
        sub = ops.pnp_ransac(packed[idx].contiguous(), P, Ks, graph_sel=sel[idx].contiguous(), flag=flags, seed=SEED,
                             return_inlier_mask=True, rng_index=idx.to(torch.int32))
        axis = 1 if isinstance(flags, tuple) else 0
        for a, b in zip(full, sub):
            assert torch.equal(a.index_select(axis, idx), b), flags
    # rng_index = 0 .. B-1 is the launch without it
    plain = ops.pnp_ransac(packed[idx].contiguous(), P, Ks, graph_sel=sel[idx].contiguous(), flag=ALL, seed=SEED)
    keyed = ops.pnp_ransac(packed[idx].contiguous(), P, Ks, graph_sel=sel[idx].contiguous(), flag=ALL, seed=SEED,
                           rng_index=torch.arange(len(idx), dtype=torch.int32, device="cuda"))
    assert all(torch.equal(a, b) for a, b in zip(plain, keyed))


@pytest.mark.parametrize("ds,objs,N", [("lmo", (1, 5, 6, 8), 512), ("ycbv", (2, 5, 15, 21), 4096), ("lm", (3, 9), 1024)])
def test_full_and_visible_poses_match_opencv(ops, ds, objs, N):
    """Each set's pose against cv2.solvePnPRansac on the same subset, on the scenes of tests/test_gpu_pnp.py: within its bars
    of OpenCV's pose, or nearer the ground truth than OpenCV's.  A subset can cost OpenCV's RANSAC more inliers than ours:
    3 of the 20 subset poses here are outside the bars that way (ycbv/15's full-mask set: OpenCV keeps 2616 inliers, we keep
    2961, the poses are 0.37 degrees apart, ours 0.16 and OpenCV's 0.52 degrees from the ground truth)."""
    B = len(objs)
    scenes = [scene(ds, o, N, 100 * o + N) for o in objs]
    scenes, packed, _, P, sel = _batch(ops, ds, objs, N, B, 300 + N, degenerate=False, scenes=scenes)
    K = torch.tensor(K_LM, dtype=torch.float32).cuda()
    R, t, n = ops.pnp_ransac(packed, P, K, graph_sel=sel, flag=(ALL, FULL, VISIB), iterations=150, seed=7)
    uv, flags, _, _, _ = ops.unpack_correspondences_host(packed)
    for v, f in enumerate((ALL, FULL, VISIB)):
        for b, (_, Rgt, tgt, _, _, _, _) in enumerate(scenes):
            X = scenes[b][0]
            valid = (flags[b] & f) != 0
            Rcv, tcv, ncv = cv2_pose(X, uv[b], valid)
            Ro, to = R[v, b].double().cpu().numpy(), t[v, b].double().cpu().numpy()
            dR, dt = rot_err_deg(Ro, Rcv), float(np.linalg.norm(to - tcv))
            print(f"{ds}/{objs[b % len(objs)]} N={N} flag {f}: valid {int(valid.sum())}, inliers ours {int(n[v, b])} / OpenCV {ncv}; "
                  f"ours vs OpenCV {dR:.3f} deg, {dt:.2f} mm; vs ground truth: ours {rot_err_deg(Ro, Rgt):.3f} deg "
                  f"{np.linalg.norm(to - tgt):.2f} mm, OpenCV {rot_err_deg(Rcv, Rgt):.3f} deg {np.linalg.norm(tcv - tgt):.2f} mm")
            nearer = rot_err_deg(Ro, Rgt) <= rot_err_deg(Rcv, Rgt) and np.linalg.norm(to - tgt) <= np.linalg.norm(tcv - tgt)
            assert (dR < TOL_R_DEG and dt < TOL_T_MM) or nearer, (f, b, dR, dt)
            assert 0.97 * ncv - 2 <= int(n[v, b]) <= int(valid.sum())
            assert rot_err_deg(Ro, Rgt) < rot_err_deg(Rcv, Rgt) + TOL_R_DEG


# ------------------------------------------------------------------------------------------------ public interface
THREE = (ALL, FULL, VISIB)


def _check_three(res3, singles):
    """forward_with_pose with flag=THREE against the three single-flag calls."""
    out3, pk3, R3, t3, n3 = res3
    for v, (out, pk, R, t, n) in enumerate(singles):
        assert torch.equal(pk3, pk) and all(torch.equal(a, b) for a, b in zip(out3, out))
        assert torch.equal(R3[v], R) and torch.equal(t3[v], t) and torch.equal(n3[v], n), f"set {v}"


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_forward_with_pose_three_sets_single_net(dtype):
    from checkerpose_b200 import head
    from checkerpose_b200.model import init, pipeline
    from checkerpose_b200.model.backbone import FeatureListBackbone
    N, B = 256, 5
    g = torch.Generator().manual_seed(8)
    xyz = syn.load_fps_xyz("lmo", 6, N)
    p3d = syn.p3d_normed_tensor(xyz).cuda()
    inet = init.InitNet_GNN(npoint=N, p3d_normed=p3d, res_log2=3, backbone_name="hrnet_w18", pretrain_backbone=False,
                            img_backbone=FeatureListBackbone())
    net = pipeline.PoseNet_GNNskip(inet, npoint=N, p3d_normed=p3d, res_log2=6, local_k=2, num_graph_module=3)
    net.load_state_dict(syn.synthetic_state_dict(syn.head_param_spec(N), g), strict=True)
    net = net.cuda().eval()
    feats = [f.cuda() for f in syn.synthetic_features(B, g)]
    bbox = syn.synthetic_bboxes(B, g).cuda()
    X = torch.tensor(xyz, dtype=torch.float32).view(1, N, 3).cuda()
    head.set_compute_dtype(dtype)
    try:
        for K in (torch.tensor(K_LM, dtype=torch.float32).cuda(), _cams(B, 9)):
            res3 = net.forward_with_pose(feats, p3d.expand(B, -1, -1), bbox, X, K, flag=THREE, seed=3)
            assert res3[2].shape == (3, B, 3, 3) and res3[3].shape == (3, B, 3) and res3[4].shape == (3, B)
            _check_three(res3, [net.forward_with_pose(feats, p3d.expand(B, -1, -1), bbox, X, K, flag=f, seed=3) for f in THREE])
    finally:
        head.set_compute_dtype(torch.float32)


def test_forward_with_pose_three_sets_lm_net():
    from checkerpose_b200 import head
    from checkerpose_b200.model import init_lm, pipeline_lm
    from checkerpose_b200.model.backbone import FeatureListBackbone
    N, B, objs = 512, 7, (1, 4, 9, 13)
    g = torch.Generator().manual_seed(21)
    p3d_all = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz("lm", o, N)) for o in objs]).cuda()
    xyz = torch.tensor(np.stack([syn.load_fps_xyz("lm", o, N) for o in objs]), dtype=torch.float32).cuda()
    inet = init_lm.InitNet_GNN(npoint=N, p3d_normed=p3d_all, res_log2=3, backbone_name="hrnet_w18", pretrain_backbone=False,
                               num_conv1x1=1, max_batch_size=8, num_graph_module=2, graph_k=20, img_backbone=FeatureListBackbone())
    net = pipeline_lm.PoseNet_GNNskip(inet, npoint=N, p3d_normed=p3d_all, res_log2=6, local_k=2, num_graph_module=3, graph_k=20)
    net.load_state_dict(syn.synthetic_state_dict(syn.head_param_spec(N), g), strict=True)
    net = net.cuda().eval()
    feats = [f.cuda() for f in syn.synthetic_features(B, g)]
    bbox = syn.synthetic_bboxes(B, g).cuda()
    obj_ids = torch.tensor([3, 1, 4, 1, 2, 4, 3]).cuda()          # 1-based index of the RoI's graph / cloud
    head.set_compute_dtype(torch.bfloat16)
    try:
        K = torch.tensor(K_LM, dtype=torch.float32).cuda()
        res3 = net.forward_with_pose(feats, None, bbox, xyz, K, obj_ids=obj_ids, flag=THREE, seed=4)
        _check_three(res3, [net.forward_with_pose(feats, None, bbox, xyz, K, obj_ids=obj_ids, flag=f, seed=4) for f in THREE])
    finally:
        head.set_compute_dtype(torch.float32)


def _bank_nets(N):
    """4 LM-O and 5 YCB-V objects in one bank (YCB-V keys offset by 100), each with its own seeded weights."""
    from test_gpu_object_bank import _build_nets
    nets = _build_nets("lmo", (1, 5, 8, 12), N, 100)
    nets.update({100 + o: n for o, n in _build_nets("ycbv", (2, 6, 11, 15, 20), N, 200).items()})
    clouds = [syn.load_fps_xyz("lmo", o, N) for o in (1, 5, 8, 12)] + [syn.load_fps_xyz("ycbv", o, N) for o in (2, 6, 11, 15, 20)]
    return nets, torch.tensor(np.stack(clouds), dtype=torch.float32).cuda()


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_object_bank_three_sets_one_launch(dtype, monkeypatch):
    from checkerpose_b200 import head, ops
    from checkerpose_b200.model.object_bank import ObjectBank
    from test_gpu_object_bank import _inputs
    N, B = 512, 40
    nets, p3d = _bank_nets(N)
    keys = sorted(nets)
    ids = torch.tensor([keys[i] for i in torch.randperm(B, generator=torch.Generator().manual_seed(12)) % len(keys)])
    ids[10:14] = 101 + 1                              # a run of one object inside the shuffle
    feats, bbox = _inputs(B, 51)
    calls = []
    for name in ("cp_pnp_ransac", "cp_pnp_ransac_sets"):
        fn = getattr(ops.lib, name)
        monkeypatch.setattr(ops.lib, name, lambda *a, _fn=fn, _name=name: calls.append(_name) or _fn(*a))
    head.set_compute_dtype(dtype)
    try:
        bank = ObjectBank(nets)
        for K in (torch.tensor(K_LM, dtype=torch.float32).cuda(), _cams(B, 17)):
            calls.clear()
            res3 = bank.forward_with_pose(feats, bbox, p3d, K, ids, flag=THREE, seed=9)
            assert calls == ["cp_pnp_ransac_sets"], calls
            single = []
            for f in THREE:
                calls.clear()
                single.append(bank.forward_with_pose(feats, bbox, p3d, K, ids, flag=f, seed=9))
                assert calls == ["cp_pnp_ransac_sets"], calls          # one launch for the batch of 9 objects
            _check_three(res3, single)
            # every RoI: its own net's forward_with_pose on the RoIs of its object
            for k, o in enumerate(keys):
                rows = torch.nonzero(ids == o).flatten().cuda()
                if len(rows) == 0:
                    continue
                Ko = K if K.dim() == 2 else K[rows]
                _, pk_o, R_o, t_o, n_o = nets[o].forward_with_pose([f[rows] for f in feats], None, bbox[rows], p3d[k:k + 1], Ko,
                                                                   flag=THREE, seed=9)
                assert torch.equal(res3[1][rows], pk_o), f"records of object {o}"
                assert torch.equal(res3[2][:, rows], R_o) and torch.equal(res3[3][:, rows], t_o) and torch.equal(res3[4][:, rows], n_o), \
                    f"poses of object {o}"
    finally:
        head.set_compute_dtype(torch.float32)
