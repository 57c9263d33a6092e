"""ms per step of the whole head (init net + 3 refine stages + decode) at several query_dims, bf16 against float32 mode.

    python scripts/kbench_widths.py [--batch 256] [--npoint 4096] [--steps 10] [--warmup 3] [--out DIR]

Weights from synthetic.head_param_spec(query_dims=...), one lmo object, synthetic HRNet features; CUDA events around
``steps`` back-to-back steps after ``warmup`` untimed ones.  Prints one JSON line per (dims, dtype) and the card's name and
power limit; with --out also writes them to DIR/kbench_widths.json."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

DIMS = [(64, 64, 64), (128, 128, 32), (96, 128, 48), (256, 256, 64), (256, 512, 128), (512, 256, 64), (512, 512, 128)]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def build(dims, N, B, dev):
    from checkerpose_b200 import synthetic as syn
    from checkerpose_b200.model import init, pipeline
    from checkerpose_b200.model.backbone import FeatureListBackbone
    g = torch.Generator().manual_seed(1234 + sum(dims))
    p3d = syn.p3d_normed_tensor(syn.load_fps_xyz("lmo", 1, N)).to(dev)
    sd = syn.synthetic_state_dict(syn.head_param_spec(N, query_dims=dims), g)
    inet = init.InitNet_GNN(npoint=N, p3d_normed=p3d, res_log2=3, backbone_name="hrnet_w18", pretrain_backbone=False,
                            max_batch_size=B, num_graph_module=2, graph_k=20, img_backbone=FeatureListBackbone())
    net = pipeline.PoseNet_GNNskip(inet, npoint=N, p3d_normed=p3d, res_log2=6, num_filters=256, max_batch_size=B,
                                   query_dims=dims, local_k=2, leaky_slope=0.01, num_graph_module=3, graph_k=20)
    net.load_state_dict(sd, strict=True)
    gg = torch.Generator(device=dev).manual_seed(4321)
    feats = [torch.relu(torch.randn(B, c, s, s, generator=gg, device=dev))
             for c, s in zip(syn.HRNET_W18_DIMS[1:], syn.HRNET_W18_SIZES[1:])]
    return net.to(dev).eval(), feats


def time_steps(net, feats, dtype, steps, warmup):
    from checkerpose_b200 import head
    f = [t.to(dtype) for t in feats]
    for _ in range(warmup):
        head.pose_head_forward(net, f, dtype=dtype)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        head.pose_head_forward(net, f, dtype=dtype)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--npoint", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("kbench_widths: no CUDA device (the numbers are GPU timings)")
    torch.set_grad_enabled(False)
    dev = torch.device("cuda")
    gpu = card()
    print(f"# {gpu}; B={args.batch} RoIs, N={args.npoint}, {args.steps} timed steps after {args.warmup}")
    rows = []
    for dims in DIMS:
        net, feats = build(dims, args.npoint, args.batch, dev)
        ms = {name: time_steps(net, feats, dt, args.steps, args.warmup)
              for name, dt in (("bf16", torch.bfloat16), ("fp32", torch.float32))}
        row = dict(query_dims="_".join(map(str, dims)), bf16_ms=round(ms["bf16"], 3), fp32_ms=round(ms["fp32"], 3),
                   fp32_over_bf16=round(ms["fp32"] / ms["bf16"], 2), batch=args.batch, npoint=args.npoint, gpu=gpu)
        print(json.dumps(row), flush=True)
        rows.append(row)
        del net, feats
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "kbench_widths.json"), "w") as fh:
            json.dump(rows, fh, indent=1)


if __name__ == "__main__":
    main()
