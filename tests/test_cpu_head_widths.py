"""Host side of the bf16 head at other query_dims, without a GPU: the zero padding of weights and BatchNorm, and the
errors for widths the kernels do not run."""
import pytest
import torch

from helpers import syn

torch.set_grad_enabled(False)


def test_pad_linear_weight_segments():
    from checkerpose_b200 import head
    g = torch.Generator().manual_seed(0)
    E, cg, d0 = 24, 96, 96
    w = torch.randn(d0, 4 * E + cg, generator=g)
    b = torch.randn(d0, generator=g)
    wp, bp = head.pad_linear_weight(w, b, ((d0, 128),), ((E, 32),) * 4 + ((cg, 128),))
    assert wp.shape == (128, 4 * 32 + 128) and bp.shape == (128,)
    for t in range(4):                     # tap t's E columns move to t * 32, the 8 after them are zero
        assert torch.equal(wp[:d0, t * 32:t * 32 + E], w[:, t * E:(t + 1) * E])
        assert not wp[:, t * 32 + E:(t + 1) * 32].any()
    assert torch.equal(wp[:d0, 128:128 + cg], w[:, 4 * E:]) and not wp[:, 128 + cg:].any()
    assert not wp[d0:].any() and torch.equal(bp[:d0], b) and not bp[d0:].any()
    same_w, same_b = head.pad_linear_weight(w, b, ((d0, d0),), ((4 * E + cg, 4 * E + cg),))
    assert torch.equal(same_w, w) and torch.equal(same_b, b)


def test_pad_edgeconv_folds_to_zero():
    """Padded EdgeConv channels: gamma = beta = mean = 0, var = 1, so the folded scale and shift are 0; both halves of the
    [x_j - x_i | x_i] input are padded alike."""
    from checkerpose_b200 import head
    g = torch.Generator().manual_seed(1)
    co, c = 96, 96
    w = torch.randn(co, 2 * c, 1, 1, generator=g)
    gamma, beta, mean = (torch.randn(co, generator=g) for _ in range(3))
    var = torch.rand(co, generator=g) + 0.5
    wp, gp, bp, mp, vp = head.pad_edgeconv(w, gamma, beta, mean, var)
    assert wp.shape == (128, 256) and gp.shape == bp.shape == mp.shape == vp.shape == (128,)
    assert torch.equal(wp[:co, :c], w[:, :c, 0, 0]) and torch.equal(wp[:co, 128:128 + c], w[:, c:, 0, 0])
    assert not wp[co:].any() and not wp[:, c:128].any() and not wp[:, 128 + c:].any()
    scale = gp / torch.sqrt(vp + 1e-5)
    shift = bp - mp * scale
    assert not scale[co:].any() and not shift[co:].any()
    assert torch.equal(vp[co:], torch.ones(128 - co)) and torch.equal(gp[:co], gamma) and torch.equal(vp[:co], var)


def test_pad_widths():
    from checkerpose_b200 import head
    assert [head.pad64(c) for c in (1, 64, 65, 96, 192, 500, 512)] == [64, 64, 128, 128, 192, 512, 512]
    assert [head.pad16(c) for c in (16, 24, 48, 100, 128)] == [16, 32, 48, 112, 128]


def _refine(dims, num_filters=256):
    from checkerpose_b200.model import pipeline
    p3d = syn.p3d_normed_tensor(syn.load_fps_xyz("ycbv", 21, 128))
    return pipeline.Refine_moduleGNN(npoint=128, p3d_normed=p3d, num_filters=num_filters, query_dims=dims, local_k=2,
                                     num_graph_module=3, graph_feat_dim=(dims or (num_filters,))[0]).eval()


@pytest.mark.parametrize("dims,what", [((640, 256, 64), "query_dims\\[0\\] up to 512 channels \\(got 640\\)"),
                                       ((256, 1024, 64), "up to 512 channels \\(got 1024\\)"),
                                       ((256, 256, 640), "up to 512 channels \\(got 640\\)"),
                                       ((98, 128, 64), "divisible by 4.*98")])
def test_bf16_width_errors(dims, what):
    from checkerpose_b200 import head
    with pytest.raises(RuntimeError, match=what) as ei:
        head.check_bf16_refine_widths(_refine(dims))
    assert "float32 mode" in str(ei.value)


@pytest.mark.parametrize("dims", [(64, 64, 64), (96, 128, 48), (512, 512, 128), (256, 256, 64)])
def test_bf16_widths_accepted(dims):
    from checkerpose_b200 import head
    head.check_bf16_refine_widths(_refine(dims))


@pytest.mark.parametrize("num_filters", [128])
def test_bf16_num_filters_accepted(num_filters):
    """num_filters sets the image branch and, with the default query_dims (num_filters, 256, 64), query_dims[0]: the bf16
    refine stage takes it (test_gpu_head_widths.py runs such a head against the oracle)."""
    from checkerpose_b200 import head
    head.check_bf16_refine_widths(_refine(None, num_filters))
