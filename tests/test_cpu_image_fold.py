"""The BatchNorm fold of the image branch (head.image_layers), checked on the CPU in float64 against each block's own
eval() forward.  All three image-branch executors (cuDNN, float32 cp_gemm_x3, bf16 slab) build from this one fold."""
import copy

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from checkerpose_b200 import head, ops
from checkerpose_b200.model import pipeline


def _randomise(module, gen):
    """He-normal weights, small biases, BatchNorm statistics with about half of the scales negative."""
    for m in module.modules():
        if isinstance(m, (nn.Conv2d, nn.ConvTranspose2d)):
            fan_in = m.weight[0].numel()
            m.weight.data = torch.randn(m.weight.shape, generator=gen) * (2.0 / fan_in) ** 0.5
            if m.bias is not None:
                m.bias.data = torch.randn(m.bias.shape, generator=gen) * 0.1
        elif isinstance(m, nn.BatchNorm2d):
            n = m.num_features
            sign = torch.where(torch.rand(n, generator=gen) < 0.5, -1.0, 1.0)
            m.weight.data = sign * (0.5 + torch.rand(n, generator=gen))
            m.bias.data = torch.randn(n, generator=gen) * 0.1
            m.running_mean = torch.randn(n, generator=gen) * 0.1
            m.running_var = 0.5 + torch.rand(n, generator=gen)
    return module.eval()


def _run_folded(layers, x):
    """The folded layers of head.image_layers in float64."""
    for kind, w, b, m, relu in layers:
        b = None if b is None else b.double()
        if kind == "conv":
            x = F.conv2d(x, w.double(), b, m.stride, m.padding, m.dilation, m.groups)
        elif kind == "convT":
            x = F.conv_transpose2d(x, w.double(), b, m.stride, m.padding, m.output_padding, m.groups, m.dilation)
        elif kind == "relu":
            x = torch.relu(x)
        elif kind == "lrelu":
            x = F.leaky_relu(x, m.negative_slope)
        else:
            x = F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=True)
        if relu:
            x = torch.relu(x)
    return x


# (name, block, input channels, input size): the image-branch blocks of PoseNet_GNNskip / InitNet_GNN at small widths
BLOCKS = [
    ("up_net[0]", lambda: pipeline.get_gdrn_upsample_module(is_convtrans=True, in_channels=96, num_filters=64), 96, 4),
    ("up_net[1]", lambda: pipeline.get_gdrn_upsample_module(is_convtrans=False, in_channels=64 + 32, num_filters=64), 96, 8),
    ("patch_generator", lambda: nn.Conv2d(64, 16, kernel_size=2, stride=1, padding=1), 64, 16),
    ("seg_block", lambda: nn.Conv2d(64, 2, kernel_size=1, padding=0, bias=True), 64, 16),
    ("conv1x1", lambda: nn.Conv2d(128, 96, kernel_size=1, stride=1, padding=0), 128, 4),
    ("conv1x1 x2", lambda: nn.Sequential(nn.Conv2d(128, 96, 1), nn.LeakyReLU(0.01), nn.Conv2d(96, 96, 1)), 128, 4),
]


@pytest.mark.parametrize("name,make,cin,size", BLOCKS, ids=[b[0] for b in BLOCKS])
def test_folded_image_block_matches_its_eval_forward(name, make, cin, size):
    gen = torch.Generator().manual_seed(7)
    block = _randomise(make(), gen)
    scales = [m.weight for m in block.modules() if isinstance(m, nn.BatchNorm2d)]
    assert all((s < 0).any() and (s > 0).any() for s in scales)
    x = torch.relu(torch.randn(2, cin, size, size, generator=gen, dtype=torch.float64))
    with torch.no_grad():
        want = copy.deepcopy(block).double()(x)
        got = _run_folded(head.image_layers(block), x)
    assert got.shape == want.shape
    err = (got - want).abs().max().item() / want.abs().max().item()
    assert err < 1e-5, f"{name}: folded layers differ from the module by {err:.2e} (relative to its largest output)"


def test_image_layers_fuse_relu_and_keep_the_other_layers():
    block = _randomise(pipeline.get_gdrn_upsample_module(is_convtrans=False, in_channels=96, num_filters=64), torch.Generator().manual_seed(1))
    assert [(k, relu) for k, _, _, _, relu in head.image_layers(block)] == [("up", False), ("conv", True), ("conv", True)]


def test_image_layers_reject_what_no_executor_runs():
    with pytest.raises(RuntimeError, match="unsupported layer in image branch: MaxPool2d"):
        head.image_layers(nn.Sequential(nn.Conv2d(8, 8, 3, padding=1), nn.MaxPool2d(2)))
    with pytest.raises(RuntimeError, match="scale_factor=2"):
        head.image_layers(nn.UpsamplingBilinear2d(scale_factor=4))


@pytest.mark.parametrize("mode,pack", [("float32", ops.pack_weight_split), ("bf16", ops.pack_weight)])
def test_own_kernel_branches_name_their_mode_when_they_reject_a_layer(mode, pack):
    """The implicit-GEMM executors take stride-1 convolutions and ReLU; the walk also accepts what only cuDNN runs."""
    for m in (nn.Conv2d(64, 64, 3, stride=2, padding=1), nn.Conv2d(64, 64, 3, padding=2, dilation=2), nn.LeakyReLU(0.01)):
        assert head.image_layers(m)
        with pytest.raises(RuntimeError, match=f"^{mode} image branch: unsupported layer"):
            head._gemm_layers(m, pack, mode)
