"""Micro-benchmark of the fused kernels at the benchmark shapes (256 RoIs, N=4096, K=20, C=256), for kernel A/B
experiments: CHECKERPOSE_B200_LIB=<variant .so> python scripts/kbench.py [k2] [k3] [chain]
Prints the average launch time (CUDA events, 20 launches after 3 warm-ups) and a checksum of the output."""
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import torch  # noqa: E402

from checkerpose_b200 import ops, synthetic as syn  # noqa: E402


def timed(fn, n=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def checksum(t):
    return float(t.float().abs().sum().item()), int(torch.isfinite(t.float()).all().item())


def main():
    what = set(sys.argv[1:]) or {"k2", "k3", "chain"}
    B, N, K, C = int(os.environ.get("KB_B", 256)), 4096, 20, 256
    g = torch.Generator().manual_seed(7)
    dev = torch.device("cuda", 0)
    p3d = syn.p3d_normed_tensor(syn.load_fps_xyz("lmo", 1, N))
    _, idx32 = ops.knn(p3d.to(dev), K, want_i32=True)
    plan = ops.GraphPlan(idx32, p3d)
    tag = os.path.basename(os.environ.get("CHECKERPOSE_B200_LIB", "default"))

    def mk(*shape, scale=1.0):
        return (torch.randn(*shape, generator=g) * scale).to(torch.bfloat16).to(dev)

    if "k2" in what:
        z = mk(B, N, 2 * C)
        w = torch.randn(2 * C, C, generator=g) / C ** 0.5
        layer = ops.chain_layer(ops.pack_weight(w.to(dev)), torch.cat([torch.zeros(C), torch.randn(C, generator=g)]).to(dev), C, 2 * C, False, 0.0)
        out = torch.empty((B, N, 2 * C), dtype=torch.bfloat16, device=dev)
        t = timed(lambda: ops.edgeconv_fwd(z=z, plan=plan, graph_sel=None, agg_slope=0.2, layer=layer, out=out, out_mode=ops.OUT_BF16))
        print(f"[{tag}] K2 256->[P|Q]512      {t:.4f} ms/launch  checksum {checksum(out)}")
        wq = torch.randn(C, C, generator=g) / C ** 0.5
        layer_q = ops.chain_layer(ops.pack_weight(wq.to(dev)), torch.randn(C, generator=g).to(dev), C, C, True, 0.01)
        a_out = torch.empty((B, N, C), dtype=torch.bfloat16, device=dev)
        hq = torch.empty((B, N, C), dtype=torch.bfloat16, device=dev)
        t = timed(lambda: ops.edgeconv_fwd(z=z, plan=plan, graph_sel=None, agg_slope=0.2, layer=layer_q, out=hq, out_mode=ops.OUT_BF16, a_out=a_out))
        print(f"[{tag}] K2 256->256 + a_out    {t:.4f} ms/launch  checksum {checksum(hq)} {checksum(a_out)}")
    if "k3" in what:
        H = 64
        patches = mk(B, H + 1, H + 1, 64)
        gf = mk(B, N, C)
        x_id = torch.randint(0, H // 2, (B, N), generator=g).to(dev)
        y_id = torch.randint(0, H // 2, (B, N), generator=g).to(dev)
        mask = (torch.rand(B, N, generator=g) > 0.2).float().to(dev)
        dims = ((256, 512), (256, 256), (512, 256))
        layers = [ops.chain_layer(ops.pack_weight((torch.randn(o, i, generator=g) * (2.0 / i) ** 0.5).to(dev)),
                                  (torch.randn(o, generator=g) * 0.1).to(dev), i, o, li < 2, 0.01) for li, (o, i) in enumerate(dims)]
        out = torch.empty((B, N, 512), dtype=torch.bfloat16, device=dev)
        t = timed(lambda: ops.chain_fwd(prologue=ops.PRO_TAPS, B=B, N=N, patches=patches, tap_step=2, x_id=x_id, y_id=y_id, mask=mask,
                                        graph_feat=gf, layers=layers, out=out, out_mode=ops.OUT_BF16))
        print(f"[{tag}] K3 taps|gf256->256->256->512  {t:.4f} ms/launch  checksum {checksum(out)}")
    if "chain" in what:
        hq = mk(B, N, C)
        dims = ((64, 256), (2, 64))
        layers = [ops.chain_layer(ops.pack_weight((torch.randn(o, i, generator=g) * (2.0 / i) ** 0.5).to(dev)),
                                  (torch.randn(o, generator=g) * 0.1).to(dev), i, o, li < 1, 0.01) for li, (o, i) in enumerate(dims)]
        logits = torch.empty((B, N, 16), dtype=torch.float32, device=dev)
        t = timed(lambda: ops.chain_fwd(prologue=ops.PRO_LOAD, B=B, N=N, src=hq, layers=layers, out=logits, out_mode=ops.OUT_F32, n_valid=2))
        print(f"[{tag}] chain 256->64->2 (query tail)  {t:.4f} ms/launch  checksum {checksum(logits[:, :, :2])}")


if __name__ == "__main__":
    main()
