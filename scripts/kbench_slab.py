"""Slab convolution (cp_conv_slab) at the image-branch shapes of the benchmark configuration: error against float64 on a
small case (single CTAs or CTA pairs, as CP_SLAB_PAIR selects), then time next to the
gather kernel cp_conv_bf16 and cuDNN: python scripts/kbench_slab.py"""
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from checkerpose_b200 import ops  # noqa: E402
from kbench_conv import timed  # noqa: E402


def padded(x):
    return ops.to_bordered(x).contiguous()


def check(dev, g):
    B, H, Cin, Cout = 5, 16, 128, 256
    x = torch.randn(B, H, H, Cin, generator=g, device=dev).to(torch.bfloat16)
    for name, k, cout in (("same3x3", 3, Cout), ("full2x2", 2, 64), ("convT", 3, Cout)):
        if name == "convT":
            w = torch.randn(Cin, cout, 3, 3, generator=g, device=dev) / (9 * Cin) ** 0.5
            wm = w.permute(1, 2, 3, 0).reshape(cout, -1).contiguous()
        else:
            w = torch.randn(cout, Cin, k, k, generator=g, device=dev) / (k * k * Cin) ** 0.5
            wm = w.permute(0, 2, 3, 1).reshape(cout, -1).contiguous()
        bias = torch.randn(cout, generator=g, device=dev)
        wp = ops.pack_weight(wm)
        xd = x.double().permute(0, 3, 1, 2)
        wd = w.to(torch.bfloat16).double()
        if name == "same3x3":
            ref = torch.relu(F.conv2d(xd, wd, bias.double(), padding=1))
            y = ops.conv_slab_same(padded(x), wp, cout, 3, 3, bias, True, 0.0)
            border = y.clone()
            border[:, :-1, :-1] = 0
            got = y[:, :-1, :-1]
            extra = f" border max {border.abs().max().item():.1e}"
        elif name == "full2x2":
            ref = torch.relu(F.conv2d(xd, wd, bias.double(), padding=1))
            got = ops.conv_slab_full(padded(x), wp, cout, 2, 2, bias, True, 0.0)
            extra = ""
        else:
            ref = torch.relu(F.conv_transpose2d(xd, wd, bias.double(), stride=2, padding=1, output_padding=1))
            y = ops.convT_slab(x, wp, cout, bias, True, 0.0)
            border = y.clone()
            border[:, :-1, :-1] = 0
            got = y[:, :-1, :-1]
            extra = f" border max {border.abs().max().item():.1e}"
        err = (got.double() - ref.permute(0, 2, 3, 1)).abs().max().item()
        print(f"  {name}: max err {err:.3e} (scale {ref.abs().max().item():.2f}){extra}")


def main():
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(3)
    print(f"variant pair={os.environ.get('CP_SLAB_PAIR', '1')}")
    check(dev, g)
    if os.environ.get("KB_CHECK_ONLY"):
        return
    B = int(os.environ.get("KB_B", 256))
    shapes = ((64, 512, 256, 3), (64, 256, 256, 3), (32, 768, 256, 3), (32, 256, 256, 3), (16, 256, 256, 3), (64, 256, 64, 2))
    if os.environ.get("KB_SHAPES"):
        shapes = ((32, 256, 256, 3), (64, 256, 64, 2))
    for H, Cin, Cout, k in shapes:
        x = torch.randn(B, H, H, Cin, generator=g, device=dev).to(torch.bfloat16)
        w = torch.randn(Cout, Cin, k, k, generator=g, device=dev) / (k * k * Cin) ** 0.5
        bias = torch.randn(Cout, generator=g, device=dev)
        wp = ops.pack_weight(w.permute(0, 2, 3, 1).reshape(Cout, -1).contiguous())
        xp = padded(x)
        Ho = H + 2 - k + 1
        if k == 3:
            ts = timed(lambda: ops.conv_slab_same(xp, wp, Cout, 3, 3, bias, True, 0.0))
        else:
            ts = timed(lambda: ops.conv_slab_full(xp, wp, Cout, 2, 2, bias, True, 0.0))
        t = timed(lambda: ops.conv_bf16(x, wp, Cout, k, k, 1, Ho, Ho, bias, True, 0.0))
        xc = x.permute(0, 3, 1, 2)
        wc = w.to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        bc = bias.to(torch.bfloat16)
        tc = timed(lambda: torch.relu_(F.conv2d(xc, wc, bc, padding=1)))
        fl = 2.0 * B * Ho * Ho * k * k * Cin * Cout
        print(f"conv{k}x{k} B={B} H={H} {Cin}->{Cout}: slab {ts:.3f} ms ({fl / ts / 1e9:.0f} TFLOP/s)   gather {t:.3f} ms ({fl / t / 1e9:.0f})   "
              f"cuDNN {tc:.3f} ms ({fl / tc / 1e9:.0f})")
    # the transposed convolution of the first up_net block (8 x 8 -> 16 x 16)
    for H, Cin, Cout in ((8, 1024, 256),):
        x = torch.randn(B, H, H, Cin, generator=g, device=dev).to(torch.bfloat16)
        w = torch.randn(Cin, Cout, 3, 3, generator=g, device=dev) / (9 * Cin) ** 0.5
        wp = ops.pack_weight(w.permute(1, 2, 3, 0).reshape(Cout, -1).contiguous())
        bias = torch.randn(Cout, generator=g, device=dev)
        ts = timed(lambda: ops.convT_slab(x, wp, Cout, bias, True, 0.0))
        t = timed(lambda: ops.conv_bf16(x, wp, Cout, 3, 3, 1, 2 * H, 2 * H, bias, True, 0.0, transposed=True))
        xc = x.permute(0, 3, 1, 2)
        wc = w.to(torch.bfloat16)
        tc = timed(lambda: torch.relu_(F.conv_transpose2d(xc, wc, bias.to(torch.bfloat16), stride=2, padding=1, output_padding=1)))
        print(f"convT3x3 B={B} H={H} {Cin}->{Cout}: slab (4 parities) {ts:.3f} ms   gather {t:.3f} ms   cuDNN {tc:.3f} ms")


if __name__ == "__main__":
    main()
