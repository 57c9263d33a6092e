"""knn(x, k) for C > 64 (knn_tcgen05.cu): tensor-core Gram tiles prune, exact fp32 direct differences decide.
The result must be the one the C <= 64 kernel defines: the k smallest fp32 direct-difference distances, ordered by
(d, j)."""
import pytest
import torch

from helpers import syn

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

WIDE_C = (65, 128, 256, 1000)
PLACES = ("before", "between", "after")


@pytest.fixture(scope="module")
def pl():
    from checkerpose_b200 import ops
    from checkerpose_b200.model import pipeline
    assert ops.lib.cp_device_arch() >= 100, "these kernels are built for sm_100a"
    return pipeline


def widen(x, C, value, where):
    """(B, C0, N) -> (B, C, N): the C0 channels of x in order, plus C - C0 channels equal to `value` at every point,
    placed before, between (spread over the gaps) or after the real ones."""
    B, C0, N = x.shape
    extra = C - C0
    if where == "before":
        counts = [extra] + [0] * C0
    elif where == "after":
        counts = [0] * C0 + [extra]
    else:
        counts = [0] + [extra // max(C0 - 1, 1) + (g < extra % max(C0 - 1, 1)) for g in range(max(C0 - 1, 1))] + [0]
        if C0 == 1:
            counts = [0, extra]
    parts = []
    for g, n in enumerate(counts):
        if n:
            parts.append(torch.full((B, n, N), value, dtype=x.dtype, device=x.device))
        if g < C0:
            parts.append(x[:, g:g + 1])
    y = torch.cat(parts, 1)
    assert y.shape == (B, C, N)
    return y.contiguous()


def check_constant_channels(pl, x, k, label, places=PLACES):
    """Constant channels add fmaf(0, 0, d) = d exactly: idx (order included) must equal the C <= 64 kernel's."""
    x = x.cuda()
    want = pl.knn(x, k)
    for C in WIDE_C:
        for value in (0.0, 1e3):
            for where in places:
                got = pl.knn(widen(x, C, value, where), k)
                assert torch.equal(got, want), f"{label}: C={C} constant {value} {where}"


def test_constant_channels_fps_fixtures(pl, golden):
    g = golden("knn")
    keys = [key for key in g if not key.startswith("rand")]
    assert len(keys) == 57
    for f, key in enumerate(keys):
        ds, oid, ns, ks = key.split("_")
        N, K = int(ns[1:]), int(ks[1:])
        p = syn.p3d_normed_tensor(syn.load_fps_xyz(ds, int(oid), N))
        # every fixture at every width and constant; the channel placement cycles over the fixtures
        check_constant_channels(pl, p, K, key, places=(PLACES[f % 3],))


def test_constant_channels_c16_golden(pl, golden):
    g = golden("knn")
    x = torch.from_numpy(g["rand_c16_n200_k12_x"])
    check_constant_channels(pl, x, 12, "rand_c16_n200_k12")


def test_constant_channels_c64_duplicates(pl):
    gen = torch.Generator().manual_seed(64)
    x = torch.randn(2, 64, 700, generator=gen)
    src = torch.randint(0, 700, (2, 120), generator=gen)
    dst = torch.randint(0, 700, (2, 120), generator=gen)
    for b in range(2):
        x[b][:, dst[b]] = x[b][:, src[b]]           # exact duplicates: ties broken towards the lower index
    check_constant_channels(pl, x, 20, "c64 duplicates")


def ref_dist64(x):
    """(B, N, N) squared distances in float64 (centred first: distances do not depend on a common offset)."""
    x = x.double()
    x = x - x.mean(2, keepdim=True)
    n = (x * x).sum(1)
    return (n[:, :, None] + n[:, None, :] - 2 * torch.bmm(x.transpose(1, 2), x)).clamp_min(0)


def check_against_f64(idx, x, k, tol=1e-4):
    """Sets equal the float64 top k except on rows whose k-th / (k+1)-th float64 gap is <= tol relative; returns the
    number of rows so exempted.  Also: entry 0 is the point itself, distances non-decreasing up to tol."""
    B, C, N = x.shape
    d = ref_dist64(x.cuda())                        # (B, N, N) float64 on the device
    srt, order = d.sort(dim=-1, stable=True)
    ref_set = order[:, :, :k].sort(-1)[0]
    got_set = idx.sort(-1)[0]
    differ = (ref_set != got_set).any(-1)
    if k < N:
        kth, nxt = srt[:, :, k - 1], srt[:, :, k]
        tie = (nxt - kth) <= tol * nxt.abs().clamp_min(1e-30)
    else:
        tie = torch.zeros_like(differ)
    bad = differ & ~tie
    assert int(bad.sum()) == 0, f"{int(bad.sum())} rows differ from the float64 top-{k} outside near-ties"
    assert (idx[:, :, 0] == torch.arange(N, device=idx.device)).all()
    dk = torch.gather(d, 2, idx)
    scale = dk[:, :, -1:].abs().clamp_min(1e-30)
    assert (dk[:, :, 1:] >= dk[:, :, :-1] - tol * scale).all(), "distances not non-decreasing"
    return int((differ & tie).sum())


@pytest.mark.parametrize("N", [64, 200, 1000, 4096])
@pytest.mark.parametrize("C", [65, 97, 128, 256, 512, 1000])
def test_random_features_vs_float64(pl, C, N):
    exempt = rows = 0
    for t, k in enumerate((1, 20, 40, 64)):
        if k > N:
            continue
        B = 1 + 2 * ((t + C + N) % 2)
        gen = torch.Generator(device="cuda").manual_seed(C * 10007 + N * 31 + k)
        x = torch.randn(B, C, N, generator=gen, device="cuda")
        idx = pl.knn(x, k)
        assert idx.dtype == torch.int64 and idx.shape == (B, N, k)
        exempt += check_against_f64(idx, x, k)
        rows += B * N
    print(f"C={C} N={N}: {exempt} of {rows} rows exempted as float64 near-ties")
    assert exempt <= 0.001 * rows


def test_offset_cloud(pl):
    gen = torch.Generator(device="cuda").manual_seed(7)
    x = 1000.0 + 0.01 * torch.randn(1, 128, 1000, generator=gen, device="cuda")
    idx = pl.knn(x, 20)
    exempt = check_against_f64(idx, x, 20)
    print(f"offset cloud: {exempt} of 1000 rows exempted as float64 near-ties")
    assert exempt <= 1


def test_all_equal_points(pl):
    x = torch.full((2, 128, 300), 0.37, device="cuda")
    idx = pl.knn(x, 20)
    assert torch.equal(idx, torch.arange(20, device="cuda").expand(2, 300, 20))


def test_deterministic_and_batch_independent(pl):
    gen = torch.Generator(device="cuda").manual_seed(11)
    x = torch.randn(3, 200, 777, generator=gen, device="cuda")
    a, a32 = pl.ops.knn(x, 33, want_i32=True)
    assert torch.equal(a, pl.knn(x, 33))
    assert torch.equal(a32.long(), a)
    for b in range(3):
        assert torch.equal(a[b], pl.knn(x[b:b + 1].clone(), 33)[0])


def test_graph_feature_through_dropin_api(pl):
    from oracle import checkerpose_oracle as orc
    gen = torch.Generator(device="cuda").manual_seed(5)
    x = torch.randn(2, 128, 512, generator=gen, device="cuda")
    idx = pl.knn(x, 20)
    y = pl.get_graph_feature(x, idx)
    want = orc.get_graph_feature(x.cpu(), idx.cpu())
    assert y.shape == (2, 256, 512, 20)
    assert torch.equal(y.cpu(), want)
    with pytest.raises(RuntimeError):
        pl.knn(x.cpu(), 20)             # CPU tensor: no fallback


def test_no_pairwise_buffer(pl):
    """B = 64, N = 4096: peak memory of the call is the input and the outputs, no (B, N, N) matrix."""
    gen = torch.Generator(device="cuda").manual_seed(3)
    x = torch.randn(64, 128, 4096, generator=gen, device="cuda")
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    idx = pl.knn(x, 20)
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    assert extra <= idx.numel() * 8 + (1 << 20), f"{extra} bytes allocated beyond the input"
    assert (idx[:, :, 0] == torch.arange(4096, device="cuda")).all()
