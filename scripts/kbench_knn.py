"""K1 (cp_knn) standalone: keypoint-count x graph_k sweep at C = 3 (the shipped graphs) and a generic-C case, then
wide features (C > 64, the tensor-core kernel) against the reference formula in torch and, at C = 64, the FFMA kernel.
Prints ms per graph and distance pairs per second; python scripts/kbench_knn.py"""
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


BF16_PEAK = 1663e12   # measured burst bf16 tensor rate of the B200 (DESIGN.md section 8)


def reference_knn(x, k):
    """pipeline.py:18-23 in torch: materialises the (B, N, N) matrix (fp32 bmm, TF32 off)."""
    inner = -2 * torch.matmul(x.transpose(2, 1), x)
    xx = torch.sum(x ** 2, dim=1, keepdim=True)
    return (-xx - inner - xx.transpose(2, 1)).topk(k=k, dim=-1)[1]


def wide(dev):
    torch.backends.cuda.matmul.allow_tf32 = False
    print("K1 wide features: cp_knn at C > 64 (tcgen05 Gram tiles, two passes, exact fp32 rescoring) vs the reference formula")
    print("Gram rate = 3*2*N^2*C*B / kernel time (one pass of split-bf16 MMAs; the kernel runs two)")
    print(f"{'B':>3} {'C':>5} {'N':>5} {'k':>3} {'ms/call':>9} {'Gram TF/s':>9} {'%bf16pk':>7} {'torch ms':>9} {'C=64 FFMA ms':>12}")
    g = torch.Generator(device=dev).manual_seed(2)
    for B in (1, 64):
        for N in (1024, 4096):
            for k in (20, 40):
                x64 = torch.randn(B, 64, N, generator=g, device=dev)
                t64 = timed(lambda: ops.knn(x64, k), n=5, warm=1)
                for C in (65, 128, 256, 512):
                    x = torch.randn(B, C, N, generator=g, device=dev)
                    t = timed(lambda: ops.knn(x, k), n=5, warm=1)
                    tr = timed(lambda: reference_knn(x, k), n=5, warm=1)
                    rate = 3 * 2 * N * N * C * B / (t * 1e-3)
                    print(f"{B:3d} {C:5d} {N:5d} {k:3d} {t:9.3f} {rate / 1e12:9.1f} {100 * rate / BF16_PEAK:6.1f}% {tr:9.3f} {t64:12.3f}",
                          flush=True)
                    del x
                del x64
                torch.cuda.empty_cache()


def main():
    dev = torch.device("cuda", 0)
    print("K1 cp_knn, 15 LM graphs per call (B' = 15, C = 3), fp32 direct-difference distances + warp top-k")
    print(f"{'N':>6} {'K':>4} {'ms/call':>9} {'ms/graph':>9} {'Gpairs/s':>9}")
    for N in (512, 1024, 2048, 4096):
        p = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz("lm", o, N)) for o in range(1, 16)], dim=0).to(dev)
        for K in (8, 16, 20, 32, 40):
            t = timed(lambda: ops.knn(p, K))
            print(f"{N:6d} {K:4d} {t:9.4f} {t / 15:9.4f} {15 * N * N / t / 1e6:9.1f}")
    g = torch.Generator(device=dev).manual_seed(1)
    for C, N, K in ((64, 4096, 20), (16, 2048, 12)):
        x = torch.randn(4, C, N, generator=g, device=dev)
        t = timed(lambda: ops.knn(x, K))
        print(f"generic C={C} N={N} K={K} B'=4: {t:.4f} ms/call, {4 * N * N * C * 2 / t / 1e9:.2f} TFLOP/s-equivalent of distance FMAs")
    wide(dev)


if __name__ == "__main__":
    main()
