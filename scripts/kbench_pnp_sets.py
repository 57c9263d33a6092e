"""The three validity sets of every RoI (all / full mask / visible mask, test.py:335-368) in one PnP launch, against the
launches it replaces.  Prints the card's name and power limit first.

  (a) B = 256 RoIs of the 21 YCB-V objects, N = 4096, 150 iterations (the scenes of tests/test_gpu_pnp.py with a band of
      rows cut from the full mask and a band of columns from the visible one): three cp_pnp_ransac launches against one
      cp_pnp_ransac_sets launch with V = 3;
  (b) the PnP stage of ObjectBank.forward_with_pose on the packed records of 8 LM-O RoIs and of 1024 YCB-V RoIs (N = 4096,
      bf16 head, synthetic features and seeded weights): one launch per object group with an index_select before and a
      scatter after (what the bank did before), against one launch over the batch with graph_sel and rng_index, for one flag
      and for three; then the whole forward_with_pose, head included, both ways.

Arms alternate within each repeat; ms per call = CUDA events over --steps calls, median over --repeats.  Every pair of arms is
checked for bit-identical results first."""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))
sys.path.insert(0, os.path.join(REPO, "scripts"))

from checkerpose_b200 import head, ops, synthetic as syn  # noqa: E402
from checkerpose_b200.model.object_bank import ObjectBank  # noqa: E402
from kbench_object_bank import LMO_IDS, compare, per_object_nets  # noqa: E402
from test_gpu_pnp import K_LM, scene  # noqa: E402

THREE = (ops.FLAG_ALL, ops.FLAG_FULL, ops.FLAG_VISIB)


def same(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


def kernel_case(args):
    B, N = 256, 4096
    scenes = [scene("ycbv", 1 + (i % 21), N, 1000 + i) for i in range(B)]
    p3d = torch.tensor(np.stack([s[0] for s in scenes]), dtype=torch.float32).cuda()
    roi = torch.tensor(np.stack([s[6] for s in scenes])).view(B, 1, N).cuda()
    seg = torch.ones(B, 2, 64, 64)
    seg[:, 1, :6] = -1.0
    seg[:, 0, :6] = -1.0
    seg[:, 0, :, :12] = -1.0
    bbox = torch.tensor(np.stack([s[3] for s in scenes])).cuda()
    xid = torch.tensor(np.stack([s[4] for s in scenes])).cuda()
    yid = torch.tensor(np.stack([s[5] for s in scenes])).cuda()
    packed = ops.correspondences_packed(roi, seg.cuda(), bbox, xid, yid)
    sel = torch.arange(B, dtype=torch.int32).cuda()
    K = torch.tensor(K_LM, dtype=torch.float32).cuda()

    def three():
        return [ops.pnp_ransac(packed, p3d, K, graph_sel=sel, flag=f, seed=1) for f in THREE]

    def one():
        return ops.pnp_ransac(packed, p3d, K, graph_sel=sel, flag=THREE, seed=1)

    a, b = three(), one()
    for v in range(3):
        assert same(a[v], [x[v] for x in b]), f"set {v} differs"
    compare(f"(a) {B} YCB-V RoIs, N = {N}, 150 iterations, flags (all, full, visible)",
            {"3 x cp_pnp_ransac": three, "cp_pnp_ransac_sets, V = 3": one}, args.steps, args.repeats, args.warmup)


def per_group_pnp(packed, g, p3d, cam_K, flag, seed):
    """The PnP stage of ObjectBank.forward_with_pose before the single launch: one cp_pnp_ransac launch per object group."""
    dev, B = packed.device, packed.shape[0]
    K = cam_K.reshape(-1, 3, 3)
    R = torch.empty((B, 3, 3), dtype=torch.float32, device=dev)
    t = torch.empty((B, 3), dtype=torch.float32, device=dev)
    ninl = torch.empty((B,), dtype=torch.int32, device=dev)
    for gi in np.unique(g):
        rows = torch.from_numpy(np.flatnonzero(g == gi)).to(dev)
        Kg = cam_K if K.shape[0] == 1 else K.index_select(0, rows)
        Rg, tg, ng = ops.pnp_ransac(packed.index_select(0, rows), p3d[gi:gi + 1], Kg, flag=flag, seed=seed)
        R[rows], t[rows], ninl[rows] = Rg, tg, ng
    return R, t, ninl


def one_launch_pnp(packed, g, p3d, cam_K, flag, seed):
    """ObjectBank.forward_with_pose's PnP stage: one launch over the batch (graph_sel = bank index, rng_index = index of the
    RoI among the RoIs of its object)."""
    dev = packed.device
    rank = np.empty(len(g), dtype=np.int32)
    for gi in np.unique(g):
        rank[g == gi] = np.arange(int((g == gi).sum()))
    return ops.pnp_ransac(packed, p3d, cam_K, graph_sel=torch.from_numpy(g.astype(np.int32)).to(dev), flag=flag, seed=seed,
                          rng_index=torch.from_numpy(rank).to(dev))


def bank_case(args, ds, ids, B, seed, label):
    N = 4096
    g = torch.Generator().manual_seed(seed)
    feats = [f.to(torch.bfloat16).cuda() for f in syn.synthetic_features(B, g)]
    bbox = syn.synthetic_bboxes(B, g).cuda()
    obj = torch.tensor([ids[i] for i in torch.randperm(B, generator=g) % len(ids)])
    bank = ObjectBank(per_object_nets(ds, ids, N))
    p3d = torch.tensor(np.stack([syn.load_fps_xyz(ds, o, N) for o in ids]), dtype=torch.float32).cuda()
    K = torch.tensor(K_LM, dtype=torch.float32).cuda()
    _, packed = bank.forward_with_correspondences(feats, bbox, obj, packed=True)
    gidx = bank._order(obj, B)[0]

    def loop(flags):
        return [per_group_pnp(packed, gidx, p3d, K, f, 0) for f in flags]

    def fused(flags):
        return one_launch_pnp(packed, gidx, p3d, K, flags if len(flags) > 1 else flags[0], 0)

    def whole_loop(flags):
        _, pk = bank.forward_with_correspondences(feats, bbox, obj, packed=True)
        return [per_group_pnp(pk, gidx, p3d, K, f, 0) for f in flags]

    def whole_fused(flags):
        return bank.forward_with_pose(feats, bbox, p3d, K, obj, flag=flags if len(flags) > 1 else flags[0])

    for flags in ((ops.FLAG_ALL,), THREE):
        a, b = loop(flags), fused(flags)
        if len(flags) == 1:
            assert same(a[0], b)
        else:
            for v in range(3):
                assert same(a[v], [x[v] for x in b]), f"set {v} differs"
        w = whole_fused(flags)
        assert torch.equal(w[1], packed) and same(w[2:], b)
        n = len(flags)
        compare(f"{label} PnP stage, {B} {ds.upper()} RoIs of {len(np.unique(gidx))} objects, N = {N}, {n} flag{'s' if n > 1 else ''}",
                {f"{n} x per-group loop ({len(np.unique(gidx))} launches each)": lambda: loop(flags), "one launch": lambda: fused(flags)},
                args.steps, args.repeats, args.warmup)
        compare(f"{label} whole forward_with_pose (bf16 head + PnP), {B} {ds.upper()} RoIs, {n} flag{'s' if n > 1 else ''}",
                {"head + per-group loop": lambda: whole_loop(flags), "ObjectBank.forward_with_pose": lambda: whole_fused(flags)},
                args.steps, args.repeats, args.warmup)
    del bank
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--skip-ycbv", action="store_true")
    args = ap.parse_args()
    torch.set_grad_enabled(False)
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True).stdout.strip())
    head.set_compute_dtype(torch.bfloat16)
    kernel_case(args)
    bank_case(args, "lmo", LMO_IDS, 8, 11, "(b1)")
    if not args.skip_ycbv:
        bank_case(args, "ycbv", tuple(range(1, 22)), 1024, 12, "(b2)")


if __name__ == "__main__":
    main()
