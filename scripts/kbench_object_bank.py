"""Mixed-object RoI batches through per-object nets: ObjectBank against a Python loop over the objects' nets (one sub-batch
per object, what a drop-in caller does without the bank) and, for YCB-V, against the shared-weight pipeline_lm step (one net,
21 graphs) that bench.py --config ycbv1024 measures.

  (a) 1024 RoIs of the 21 YCB-V objects: shipped FPS keypoints, N = 4096, K = 20, distinct seeded weights per object;
  (b) 8 RoIs of the 8 LM-O objects at N = 4096.

bf16 mode, tcgen05 image branch, synthetic backbone features (bf16).  Every arm returns packed correspondence records.  Arms
alternate within each repeat; ms per forward = CUDA events over --steps forwards, median over --repeats.  Prints the card's
name and power limit first."""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from checkerpose_b200 import head, synthetic as syn  # noqa: E402
from checkerpose_b200.model import init, init_lm, pipeline, pipeline_lm  # noqa: E402
from checkerpose_b200.model.backbone import FeatureListBackbone  # noqa: E402
from checkerpose_b200.model.object_bank import ObjectBank  # noqa: E402

LMO_IDS = (1, 5, 6, 8, 9, 10, 11, 12)


def build(I, P, N, p3d, seed):
    inet = I.InitNet_GNN(npoint=N, p3d_normed=p3d, res_log2=3, backbone_name="hrnet_w18", pretrain_backbone=False, num_conv1x1=1,
                         max_batch_size=8, num_graph_module=2, graph_k=20, img_backbone=FeatureListBackbone())
    net = P.PoseNet_GNNskip(inet, npoint=N, p3d_normed=p3d, res_log2=6, num_filters=256, max_batch_size=8, local_k=2, leaky_slope=0.01,
                            num_graph_module=3, graph_k=20)
    net.load_state_dict(syn.synthetic_state_dict(syn.head_param_spec(N), torch.Generator().manual_seed(seed)), strict=True)
    return net.cuda().eval()


def per_object_nets(ds, ids, N):
    return {o: build(init, pipeline, N, syn.p3d_normed_tensor(syn.load_fps_xyz(ds, o, N)).cuda(), 1000 + o) for o in ids}


def timed(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def compare(title, arms, steps, repeats, warmup):
    for fn in arms.values():
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    t = {k: [] for k in arms}
    for _ in range(repeats):
        for k, fn in arms.items():
            t[k].append(timed(fn, steps))
    print(f"\n{title}")
    base = np.median(t[next(iter(arms))])
    for k, v in t.items():
        m = np.median(v)
        print(f"  {k:<34s} {m:9.3f} ms per forward (min {min(v):.3f}, max {max(v):.3f})  x{m / base:.3f} of the first")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--skip-ycbv", action="store_true")
    args = ap.parse_args()
    torch.set_grad_enabled(False)
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True).stdout.strip())
    head.set_compute_dtype(torch.bfloat16)
    N = 4096
    cases = [("lmo", LMO_IDS, 8, 11)] + ([] if args.skip_ycbv else [("ycbv", tuple(range(1, 22)), 1024, 12)])
    for ds, ids, B, seed in cases:
        g = torch.Generator().manual_seed(seed)
        feats = [f.to(torch.bfloat16).cuda() for f in syn.synthetic_features(B, g)]
        bbox = syn.synthetic_bboxes(B, g).cuda()
        obj = torch.tensor([ids[i] for i in torch.randperm(B, generator=g) % len(ids)])
        nets = per_object_nets(ds, ids, N)
        bank = ObjectBank(nets)
        rows = {o: torch.nonzero(obj == o).flatten().cuda() for o in ids}

        def loop():
            out = []
            for o in ids:
                r = rows[o]
                if len(r):
                    out.append(nets[o].forward_with_correspondences([f.index_select(0, r) for f in feats], None, bbox.index_select(0, r), packed=True))
            return out

        arms = {"ObjectBank": lambda: bank.forward_with_correspondences(feats, bbox, obj, packed=True),
                f"loop over the {len(ids)} nets": loop}
        if ds == "ycbv":
            p3d = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz(ds, o, N)) for o in ids]).cuda()
            shared = build(init_lm, pipeline_lm, N, p3d, 7)
            obj_dev = obj.cuda()
            arms["shared-weight pipeline_lm step"] = lambda: shared.forward_with_correspondences(feats, None, bbox, obj_ids=obj_dev, packed=True)
        compare(f"({'a' if ds == 'ycbv' else 'b'}) {B} RoIs of the {len(ids)} {ds.upper()} objects, N = {N}, K = 20, bf16", arms,
                args.steps, args.repeats, args.warmup)
        del nets, bank, arms
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
