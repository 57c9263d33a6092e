"""The launches of the one-GPU ycbv1024 step at its sizes: tensors past 2^31 elements and 4 GiB.

``bench.py --config ycbv1024`` on one GPU puts 1024 RoIs through every launch: the [P|Q] tables of the EdgeConvs are
(1024, 4096, 512) bf16 = 2^31 elements, the 64 x 64 concatenation of up_net is (1024, 65, 65, 512) bf16, and with
``--dtype fp32`` the same tensors are 8 GiB.  A 32-bit offset that wraps inside such a tensor does not fault: it reads or
writes another RoI's rows.  Each case below runs one launch as head.py issues it, with the batch chosen so that element
offset 2^31 and byte offsets 2^31 and 2^32 of its largest tensor fall strictly inside the batch (B = 1100 RoIs for N = 4096
node tensors, B = 1040 for 64 x 64 maps), and checks it two ways:

(a) bit-identity: the big launch equals, on every RoI, the same launch over batch slices in which every tensor stays
    below 2 GiB -- the regime the float64 tests of test_gpu_kernels.py and test_gpu_many_tiles.py validate.  A wrapped
    offset shows up here in the RoI it corrupts and in the RoI it was meant for;
(b) float64 maths on the same rounded operands over the RoIs on both sides of every boundary, the first and the last
    RoI, at the bar of the kernel's existing test.

Inputs are made on the device from seeded generators.  Each case computes its memory need from CASES and skips, naming
the bytes, when the device has less free memory."""
import math
import subprocess

import pytest
import torch
import torch.nn.functional as F

from helpers import agg_rows, bf16r, rel_max, syn

torch.set_grad_enabled(False)
gpu = pytest.mark.gpu

GiB = 1 << 30
N = 4096
B_NODES = 1100      # (B, 4096, 512) bf16 passes 2^31 elements at RoI 1024
B_MAPS = 1040       # (B, 65, 65, 512) bf16 passes 2^31 elements at RoI 992
BF16, F32 = torch.bfloat16, torch.float32
G_YCBV = 21         # YCB-V: 21 objects = 21 graphs, one selected per RoI

# case -> (B, {tensor: (shape of one RoI, bytes per element)} of every full-batch tensor of the case, the byte offset its
# largest tensor exists to pass).  The tests build their tensors from this table and check their sizes against it.
IDS = {"x_id": ((N,), 8), "y_id": ((N,), 8), "mask": ((N,), 4)}
CASES = {
    "k3": (B_NODES, {"patches": ((65, 65, 64), 2), "graph_feat": ((N, 256), 2), **IDS, "out": ((N, 512), 2)}, 1 << 32),
    "edgeconv_pq": (B_NODES, {"z": ((N, 512), 2), "out": ((N, 512), 2)}, 1 << 32),
    "edgeconv_last": (B_NODES, {"z": ((N, 512), 2), "a_out": ((N, 256), 2), "out": ((N, 256), 2)}, 1 << 32),
    "chain_agg": (B_NODES, {"z": ((N, 512), 2), "a_out": ((N, 256), 2), "out": ((N, 512), 2)}, 1 << 32),
    "chain_load": (B_NODES, {"z": ((N, 512), 2), "out": ((N, 512), 2)}, 1 << 32),
    "query_tail": (B_NODES, {"src": ((N, 256), 2), "x_bits": ((6, N), 4), "y_bits": ((6, N), 4), "x_id": ((N,), 8),
                             "y_id": ((N,), 8), "x_id_kp": ((N,), 8), "y_id_kp": ((N,), 8), "logits": ((N, 2), 4)}, 1 << 31),
    "slab": (B_MAPS, {"x512": ((65, 65, 512), 2), "x256": ((65, 65, 256), 2), "out": ((65, 65, 256), 2),
                      "seg": ((2, 64, 64), 4)}, 1 << 32),
    "upsample": (B_MAPS, {"a_bordered": ((33, 33, 256), 2), "b": ((32, 32, 256), 2), "out": ((65, 65, 512), 2)}, 1 << 32),
    "x3_linear_pg0": (B_NODES, {"a1": ((N, 256), 4), "a2": ((N, 256), 4), "out": ((N, 256), 4)}, 1 << 32),
    "x3_linear_pq": (B_NODES, {"a1": ((N, 256), 4), "out": ((N, 512), 4)}, 1 << 32),
    "x3_conv": (B_MAPS, {"x": ((64, 64, 512), 4), "out": ((64, 64, 256), 4)}, 1 << 32),
    "agg_f32": (B_NODES, {"z": ((N, 512), 4), "out": ((N, 256), 4)}, 1 << 32),
    "taps_f32": (B_NODES, {"patches": ((65, 65, 64), 4), **IDS, "out": ((N, 256), 4)}, 1 << 32),
}
SLICE_BYTES = 1 << 31       # every tensor of a slice launch stays below this
MARGIN = 2 * GiB            # references, slice outputs of in-place buffers, graph tables


def roi_bytes(case, name):
    shape, es = CASES[case][1][name]
    return math.prod(shape) * es


def largest(case):
    B, tensors, _ = CASES[case]
    name = max(tensors, key=lambda t: roi_bytes(case, t))
    return name, B * roi_bytes(case, name)


def boundary_rois(case):
    """The first and last RoI and, for every tensor of the case, the RoIs on both sides of element offset 2^31 and of
    byte offsets 2^31 and 2^32."""
    B, tensors, _ = CASES[case]
    rois = {0, B - 1}
    for name, (_, es) in tensors.items():
        rb = roi_bytes(case, name)
        for off in (1 << 31, 1 << 32, (1 << 31) * es):
            if off < B * rb:
                rois.update({(off - 1) // rb, off // rb})
    return sorted(rois)


def slice_step(case):
    """RoIs per slice launch of oracle (a)."""
    return (SLICE_BYTES - 1) // max(roi_bytes(case, t) for t in CASES[case][1])


def peak_bytes(case):
    B, tensors, _ = CASES[case]
    per_roi = sum(roi_bytes(case, t) for t in tensors)
    return (B + slice_step(case)) * per_roi + MARGIN


# ------------------------------------------------------------------------------------------------ CPU: the table itself
def test_cases_pass_their_boundaries():
    """Each case's largest tensor passes the byte offset the case exists for (2^31 for the query tail's (B,N,256) source,
    2^32 for every other case); every boundary RoI lies strictly inside the batch, the case's own boundary among them;
    slice launches stay below 2 GiB."""
    for case, (B, tensors, bound) in CASES.items():
        name, nbytes = largest(case)
        assert nbytes > bound, f"{case}: largest tensor {name} has {nbytes} bytes, not past {bound}"
        rois = boundary_rois(case)
        inner = rois[1:-1]
        assert rois[0] == 0 and rois[-1] == B - 1
        assert inner and all(0 < r < B - 1 for r in inner), f"{case}: boundary RoIs {rois} of a batch of {B}"
        rb = roi_bytes(case, name)
        assert bound // rb in inner and (bound - 1) // rb in inner, f"{case}: byte {bound} of {name} is not inside the batch"
        step = slice_step(case)
        assert 1 <= step < B and step * max(roi_bytes(case, t) for t in tensors) < SLICE_BYTES
    assert CASES["query_tail"][2] == 1 << 31
    assert all(bound == 1 << 32 for case, (_, _, bound) in CASES.items() if case != "query_tail")


# ------------------------------------------------------------------------------------------------ GPU plumbing
def _power_limit():
    try:
        uuid = torch.cuda.get_device_properties(torch.cuda.current_device()).uuid
        res = subprocess.run(["nvidia-smi", "-i", f"GPU-{uuid}", "--query-gpu=power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60)
        return res.stdout.strip() or "not read"
    except (AttributeError, OSError, subprocess.SubprocessError):
        return "not read"


@pytest.fixture(scope="module")
def ops():
    from checkerpose_b200 import ops
    assert ops.lib.cp_device_arch() >= 100, "these kernels are built for sm_100a"
    print(f"\n[device] {torch.cuda.get_device_name()}, power limit {_power_limit()}")
    return ops


@pytest.fixture(scope="module")
def ycbv_graphs(ops):
    """K -> the (21, N, K) int32 kNN tables of the 21 YCB-V objects at N keypoints."""
    p3d = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz("ycbv", o, N)) for o in range(1, G_YCBV + 1)], dim=0).cuda()
    cache = {}

    def get(K):
        if K not in cache:
            cache[K] = ops.knn(p3d, K, want_i32=True)[1]
        return cache[K]
    get.p3d = p3d
    return get


@pytest.fixture(scope="module")
def ycbv_plan(ops, ycbv_graphs):
    """The graph plan of the benchmark's ycbv graphs (K = 20): the staged kernels run on it."""
    plan = ops.GraphPlan(ycbv_graphs(20), ycbv_graphs.p3d)
    assert plan.staged
    return plan


def need_memory(case):
    """Skip unless the device has the case's peak need free -> B."""
    torch.cuda.empty_cache()
    need = peak_bytes(case)
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"{case}: needs {need} bytes ({need / GiB:.1f} GiB) of device memory, {free / GiB:.1f} GiB free")
    torch.cuda.reset_peak_memory_stats()
    return CASES[case][0]


def gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def randn(*shape, g, dtype=F32):
    return torch.randn(shape, generator=g, device="cuda", dtype=dtype)


def bordered_randn(B, H, C, g):
    """A bordered bf16 NHWC map (B, H+1, W+1, C): random interior, zero last row and column."""
    x = torch.zeros((B, H + 1, H + 1, C), dtype=BF16, device="cuda")
    x[:, :H, :H].normal_(generator=g)
    return x


def check_size(case, name, t):
    B, tensors, _ = CASES[case]
    shape, es = tensors[name]
    assert tuple(t.shape) == (B,) + shape and t.element_size() == es, f"{case}: {name} is {tuple(t.shape)}, table says {shape}"


def _bits(t):
    return t.view({2: torch.int16, 4: torch.int32, 8: torch.int64}[t.element_size()]) if t.is_floating_point() else t


def same_bits(a, b):
    return torch.equal(_bits(a), _bits(b))


def check_slices(case, run, big):
    """Oracle (a): run(b0, b1) over slices below 2 GiB gives the bits of the big launch's outputs ``big``."""
    B = CASES[case][0]
    step = slice_step(case)
    for b0 in range(0, B, step):
        b1 = min(B, b0 + step)
        for i, (a, p) in enumerate(zip(big, run(b0, b1))):
            if not same_bits(a[b0:b1], p):
                bad = ((_bits(a[b0:b1]) != _bits(p)).flatten(1).any(1).nonzero().flatten() + b0).tolist()
                raise AssertionError(f"{case}: output {i} differs between the {B}-RoI launch and the {b1 - b0}-RoI launch of "
                                     f"RoIs {b0}-{b1 - 1} in {len(bad)} RoIs: {bad[:8]}{' ...' if len(bad) > 8 else ''}")


def rows_of(rois):
    """(b, n) of every node row of the listed RoIs, and the RoIs as a device tensor."""
    r = torch.tensor(rois, device="cuda")
    return r, r.repeat_interleave(N), torch.arange(N, device="cuda").repeat(len(rois))


def report(case, errs):
    B = CASES[case][0]
    name, nbytes = largest(case)
    shape, es = CASES[case][1][name]
    print(f"[{case}] B={B}: largest tensor {name} {(B,) + shape} of {8 * es}-bit elements = {nbytes / GiB:.2f} GiB = "
          f"{nbytes / es / 2 ** 31:.3f} x 2^31 elements; boundary RoIs {boundary_rois(case)}; {errs}; "
          f"peak allocated {torch.cuda.max_memory_allocated() / GiB:.1f} GiB")


def lrelu64(x, s):
    return torch.where(x > 0, x, x * s)


def chain_ref(x, ws, bs, acts):
    """float64 chain of Linear layers on bf16 operands, intermediates re-quantised to bf16 as the kernels store them."""
    h = x.double()
    for li, (w, b, act) in enumerate(zip(ws, bs, acts)):
        h = h @ w.double().t() + b.double()
        if act:
            h = lrelu64(h, 0.01)
        if li < len(ws) - 1:
            h = bf16r(h.float()).double()
    return h


def bf16_weights(g, dims):
    ws = [bf16r(randn(o, i, g=g) * (2.0 / i) ** 0.5) for o, i in dims]
    bs = [randn(o, g=g) * 0.1 for o, _ in dims]
    return ws, bs


# ------------------------------------------------------------------------------------------------ K3 taps chain
@gpu
def test_k3_taps_chain(ops):
    """cp_chain_fwd(CP_PRO_TAPS) as a refine stage issues it: 4-tap gather + graph feature -> (256+256) -> 256 -> 256 -> 512."""
    case = "k3"
    B = need_memory(case)
    g = gen(3)
    patches = randn(B, 65, 65, 64, g=g, dtype=BF16)
    gf = randn(B, N, 256, g=g, dtype=BF16)
    x_id = torch.randint(0, 32, (B, N), generator=g, device="cuda")
    y_id = torch.randint(0, 32, (B, N), generator=g, device="cuda")
    mask = (torch.rand(B, N, generator=g, device="cuda") > 0.2).float()
    dims, acts = ((256, 512), (256, 256), (512, 256)), (True, True, False)
    ws, bs = bf16_weights(g, dims)
    layers = [ops.chain_layer(ops.pack_weight(w), b, w.shape[1], w.shape[0], a, 0.01) for w, b, a in zip(ws, bs, acts)]

    def run(b0, b1):
        out = torch.empty((b1 - b0, N, 512), dtype=BF16, device="cuda")
        ops.chain_fwd(prologue=ops.PRO_TAPS, B=b1 - b0, N=N, tap_step=2, layers=layers, out=out, out_mode=ops.OUT_BF16,
                      patches=patches[b0:b1], x_id=x_id[b0:b1], y_id=y_id[b0:b1], mask=mask[b0:b1], graph_feat=gf[b0:b1])
        return (out,)
    big = run(0, B)
    for name, t in (("patches", patches), ("graph_feat", gf), ("x_id", x_id), ("y_id", y_id), ("mask", mask), ("out", big[0])):
        check_size(case, name, t)
    check_slices(case, run, big)
    _, bi, ni = rows_of(boundary_rois(case))
    yy, xx = 2 * y_id[bi, ni], 2 * x_id[bi, ni]
    taps = torch.cat([patches[bi, yy + dy, xx + dx] for dy, dx in ((0, 0), (2, 0), (0, 2), (2, 2))], dim=-1)
    h = chain_ref(torch.cat([taps.double() * mask[bi, ni, None].double(), gf[bi, ni].double()], dim=-1), ws, bs, acts)
    err = rel_max(big[0][bi, ni], h)
    report(case, f"float64 max err / max = {err:.2e}")
    assert err < 2e-2, err          # test_taps_chain_many_tiles' bar: three layers, intermediates re-quantised to bf16


# ------------------------------------------------------------------------------------------------ EdgeConv and the generic chain
def agg_ref(z, nb_of, rois, Co):
    """float64-exact aggregation of the listed RoIs (nb_of(r) -> (R,N,K) neighbour rows) as bf16 values, (R*N, Co)."""
    r, _, _ = rows_of(rois)
    R = len(rois)
    bi, ni = torch.arange(R, device="cuda").repeat_interleave(N), torch.arange(N, device="cuda").repeat(R)
    return agg_rows(z[r], nb_of(r), bi, ni, Co, 0.2, True)


@gpu
@pytest.mark.parametrize("form", ["pq", "last"])
def test_edgeconv(ops, ycbv_plan, form):
    """cp_edgeconv_fwd on the ycbv K = 20 plan with a graph per RoI: the aggregation fused with the next EdgeConv's [P|Q]
    GEMM 256 -> 512 ("pq"), and the last EdgeConv of a stage, 256 -> 256 with the aggregation stored ("last")."""
    case = f"edgeconv_{form}"
    B = need_memory(case)
    g = gen(20 + len(form))
    Co, nout, act = 256, (512 if form == "pq" else 256), form == "last"
    z = randn(B, N, 2 * Co, g=g, dtype=BF16)
    sel = torch.randint(0, G_YCBV, (B,), generator=g, device="cuda", dtype=torch.int32)
    (w,), (bias,) = bf16_weights(g, ((nout, Co),))
    layer = ops.chain_layer(ops.pack_weight(w), bias, Co, nout, act, 0.01)

    def run(b0, b1):
        out = torch.empty((b1 - b0, N, nout), dtype=BF16, device="cuda")
        a_out = torch.empty((b1 - b0, N, Co), dtype=BF16, device="cuda") if form == "last" else None
        ops.edgeconv_fwd(z=z[b0:b1], plan=ycbv_plan, graph_sel=sel[b0:b1], agg_slope=0.2, layer=layer, out=out,
                         out_mode=ops.OUT_BF16, a_out=a_out)
        return (out,) if a_out is None else (out, a_out)
    big = run(0, B)
    check_size(case, "z", z)
    check_size(case, "out", big[0])
    if form == "last":
        check_size(case, "a_out", big[1])
    check_slices(case, run, big)
    rois = boundary_rois(case)
    r, _, _ = rows_of(rois)
    a_ref = agg_ref(z, lambda r: ycbv_plan.idx_p[sel[r].long()].long(), rois, Co)
    if form == "last":
        assert torch.equal(big[1][r].reshape(-1, Co).float(), a_ref), "the stored aggregation must be bit-exact"
    ref = chain_ref(a_ref, [w], [bias], [act])
    got = big[0][r].reshape(-1, nout).double()
    err = rel_max(got, ref)
    report(case, f"aggregation {'bit-exact' if form == 'last' else 'not stored'}, GEMM float64 max err / max = {err:.2e}")
    assert torch.allclose(got, ref, rtol=1e-2, atol=1e-2), err


@gpu
@pytest.mark.parametrize("prologue", ["agg", "load"])
def test_chain(ops, ycbv_graphs, prologue):
    """cp_chain_fwd(CP_PRO_AGG): the head's EdgeConv where the staged kernel does not fit (K = 41 here), aggregation
    stored and 256 -> 512; cp_chain_fwd(CP_PRO_LOAD) over the Q half of the same table (row stride 512), 256 -> 512."""
    case = f"chain_{prologue}"
    B = need_memory(case)
    g = gen(41 + len(prologue))
    Co, nout = 256, 512
    z = randn(B, N, 2 * Co, g=g, dtype=BF16)
    (w,), (bias,) = bf16_weights(g, ((nout, Co),))
    layer = ops.chain_layer(ops.pack_weight(w), bias, Co, nout, True, 0.01)
    rois = boundary_rois(case)
    r, _, _ = rows_of(rois)
    if prologue == "agg":
        idx32 = ycbv_graphs(41)
        sel = torch.randint(0, G_YCBV, (B,), generator=g, device="cuda", dtype=torch.int32)

        def run(b0, b1):
            a_out = torch.empty((b1 - b0, N, Co), dtype=BF16, device="cuda")
            out = torch.empty((b1 - b0, N, nout), dtype=BF16, device="cuda")
            ops.chain_fwd(prologue=ops.PRO_AGG, B=b1 - b0, N=N, z=z[b0:b1], idx32=idx32, graph_sel=sel[b0:b1], agg_slope=0.2,
                          a_out=a_out, layers=[layer], out=out, out_mode=ops.OUT_BF16)
            return out, a_out
        big = run(0, B)
        check_size(case, "a_out", big[1])
        a_ref = agg_ref(z, lambda r: idx32[sel[r].long()].long(), rois, Co)
        assert torch.equal(big[1][r].reshape(-1, Co).float(), a_ref), "the stored aggregation must be bit-exact"
        x, note = a_ref, "aggregation bit-exact"
    else:
        src = z[..., Co:]

        def run(b0, b1):
            out = torch.empty((b1 - b0, N, nout), dtype=BF16, device="cuda")
            ops.chain_fwd(prologue=ops.PRO_LOAD, B=b1 - b0, N=N, src=src[b0:b1], layers=[layer], out=out, out_mode=ops.OUT_BF16)
            return (out,)
        big = run(0, B)
        x, note = src[r].reshape(-1, Co), "source rows of stride 512"
    check_size(case, "z", z)
    check_size(case, "out", big[0])
    check_slices(case, run, big)
    ref = chain_ref(x, [w], [bias], [True])
    got = big[0][r].reshape(-1, nout).double()
    err = rel_max(got, ref)
    report(case, f"{note}, GEMM float64 max err / max = {err:.2e}")
    assert torch.allclose(got, ref, rtol=1e-2, atol=1e-2), err


# ------------------------------------------------------------------------------------------------ query tail + decode
@gpu
def test_query_tail(ops, ycbv_plan):
    """cp_query_decode_fwd as the last refine stage issues it: src (B,N,256) -> 64 -> 2 logits, decoded into bit plane 4 of
    6 through the plan permutation of each RoI's graph, ids updated in place and written in keypoint order."""
    case = "query_tail"
    B = need_memory(case)
    g = gen(64)
    kin, Ltot, plane = 256, 6, 4
    src = randn(B, N, kin, g=g, dtype=BF16)
    w1 = bf16r(randn(64, kin, g=g) / kin ** 0.5)
    b1 = randn(64, g=g) * 0.1
    w2 = randn(2, 64, g=g) / 8.0
    b2 = randn(2, g=g) * 0.1
    perm = ycbv_plan.perm
    sel = torch.randint(0, G_YCBV, (B,), generator=g, device="cuda", dtype=torch.int32)
    x_id0 = torch.randint(0, 16, (B, N), generator=g, device="cuda")
    y_id0 = torch.randint(0, 16, (B, N), generator=g, device="cuda")
    w1p = ops.pack_weight(w1)
    nan = float("nan")

    def buffers():
        return dict(x_bits=torch.full((B, Ltot, N), nan, device="cuda"), y_bits=torch.full((B, Ltot, N), nan, device="cuda"),
                    x_id=x_id0.clone(), y_id=y_id0.clone(), logits=torch.zeros((B, N, 2), device="cuda"),
                    x_id_kp=torch.full((B, N), -1, dtype=torch.int64, device="cuda"),
                    y_id_kp=torch.full((B, N), -1, dtype=torch.int64, device="cuda"))

    def run(b0, b1_, d):
        ops.query_decode_fwd(src=src[b0:b1_], w1_packed=w1p, b1=b1, slope=0.01, w2=w2, b2=b2, plane=plane, Ltot=Ltot,
                             perm=perm, graph_sel=sel[b0:b1_], **{k: v[b0:b1_] for k, v in d.items()})
    big = buffers()
    run(0, B, big)
    check_size(case, "src", src)
    for k, v in big.items():
        check_size(case, k, v)
    small = buffers()
    step = slice_step(case)
    for b0 in range(0, B, step):
        run(b0, min(B, b0 + step), small)
    for k in big:
        assert same_bits(big[k], small[k]), f"{case}: {k} of the {B}-RoI launch differs from {step}-RoI launches"
    lg = big["logits"]
    r, _, _ = rows_of(boundary_rois(case))
    ref = lrelu64(src[r].double() @ w1.double().t() + b1.double(), 0.01) @ w2.double().t() + b2.double()
    err = rel_max(lg[r], ref)
    # the decode of the kernel's own logits, exactly, on every row
    kp = perm[sel.long()].long()
    want_x = torch.full((B, N), nan, device="cuda").scatter_(1, kp, lg[..., 0])
    want_y = torch.full((B, N), nan, device="cuda").scatter_(1, kp, lg[..., 1])
    xb, yb = big["x_bits"], big["y_bits"]
    assert torch.equal(xb[:, plane], want_x) and torch.equal(yb[:, plane], want_y), "decoded bit planes differ"
    others = [p for p in range(Ltot) if p != plane]
    assert bool(torch.isnan(xb[:, others]).all()) and bool(torch.isnan(yb[:, others]).all()), "other bit planes were written"
    nx, ny = x_id0 * 2 + (lg[..., 0] > 0).long(), y_id0 * 2 + (lg[..., 1] > 0).long()
    assert torch.equal(big["x_id"], nx) and torch.equal(big["y_id"], ny), "updated ids differ"
    zeros = torch.zeros((B, N), dtype=torch.int64, device="cuda")
    assert torch.equal(big["x_id_kp"], zeros.scatter(1, kp, nx)) and torch.equal(big["y_id_kp"], zeros.scatter(1, kp, ny)), \
        "keypoint-order ids differ"
    report(case, f"logits float64 max err / max = {err:.2e}, bits and ids exact on every row")
    assert err < 1e-3, err


# ------------------------------------------------------------------------------------------------ image branch (bf16)
@gpu
def test_slab_convs(ops, monkeypatch):
    """cp_conv_slab over bordered 64 x 64 maps as up_net[2] and patch_generator issue it: 3x3 512 -> 256 on the concat,
    3x3 256 -> 256 with the fused seg head, 2x2 (padding 1) 256 -> 64; CTA pairs and single CTAs."""
    case = "slab"
    B = need_memory(case)
    g = gen(512)
    x512 = bordered_randn(B, 64, 512, g)
    x256 = bordered_randn(B, 64, 256, g)
    check_size(case, "x512", x512)
    check_size(case, "x256", x256)
    seg = ((randn(2, 256, g=g) / 16.0).contiguous(), randn(2, g=g))
    rois = boundary_rois(case)
    r = torch.tensor(rois, device="cuda")
    errs = []
    for kind, x, k, cout in (("same3 512->256", x512, 3, 256), ("same3 256->256 + seg", x256, 3, 256), ("full2 256->64", x256, 2, 64)):
        cin = x.shape[-1]
        w = bf16r(randn(cout, cin, k, k, g=g) / (cin * k * k) ** 0.5)
        bias = randn(cout, g=g)
        wp = ops.pack_weight(w.permute(0, 2, 3, 1).reshape(cout, k * k * cin).contiguous())
        full, with_seg = k == 2, "seg" in kind

        def run(b0, b1):
            if full:
                return (ops.conv_slab_full(x[b0:b1], wp, cout, 2, 2, bias, True, 0.0),)
            if with_seg:
                return ops.conv_slab_same(x[b0:b1], wp, cout, 3, 3, bias, True, 0.0, seg=seg)
            return (ops.conv_slab_same(x[b0:b1], wp, cout, 3, 3, bias, True, 0.0),)
        xs = x[r, :64, :64].permute(0, 3, 1, 2).double()
        ref = torch.relu(F.conv2d(xs, w.double(), bias.double(), padding=1)).permute(0, 2, 3, 1)
        for pair in ("1", "0"):
            monkeypatch.setenv("CP_SLAB_PAIR", pair)
            big = run(0, B)
            if cout == 256:
                check_size(case, "out", big[0])
            if with_seg:
                check_size(case, "seg", big[1])
            check_slices(case, run, big)
            out = big[0][r]
            if not full:
                assert not bool(big[0][:, -1].any()) and not bool(big[0][:, :, -1].any()), f"{kind}: border not zero"
                out = out[:, :-1, :-1]
            err = rel_max(out, ref)
            errs.append(f"{kind} pair={pair} {err:.2e}")
            assert err < 6e-3, (kind, pair, err)
            if with_seg:
                sref = torch.einsum("bhwc,jc->bjhw", out.double(), seg[0].double()) + seg[1].double().view(1, -1, 1, 1)
                serr = rel_max(big[1][r], sref)
                errs.append(f"seg head {serr:.2e}")
                assert serr < 1e-5, (kind, pair, serr)
            del big, out
    report(case, "float64 max err / max: " + ", ".join(errs))


@gpu
def test_upsample2x_cat_padded(ops):
    """cp_zero_border_nhwc + cp_upsample2x_cat_nhwc_to as up_net[2] issues them: two (B,256,32,32) maps, the first the
    interior view of a bordered buffer -> the bordered (B,65,65,512) concat."""
    case = "upsample"
    B = need_memory(case)
    g = gen(65)
    a_bordered = bordered_randn(B, 32, 256, g)
    a = a_bordered[:, :32, :32].permute(0, 3, 1, 2)
    b = randn(B, 32, 32, 256, g=g, dtype=BF16).permute(0, 3, 1, 2)

    def run(b0, b1):
        return (ops.upsample2x_cat_padded(a[b0:b1], b[b0:b1]),)
    big = run(0, B)
    check_size(case, "a_bordered", a_bordered)
    check_size(case, "b", b.permute(0, 2, 3, 1))
    check_size(case, "out", big[0])
    check_slices(case, run, big)
    out = big[0]
    assert not bool(out[:, -1].any()) and not bool(out[:, :, -1].any()), "border not zero"
    r = torch.tensor(boundary_rois(case), device="cuda")
    ref = F.interpolate(torch.cat([a[r], b[r]], 1).double(), scale_factor=2, mode="bilinear", align_corners=True)
    got = out[r, :-1, :-1].permute(0, 3, 1, 2).double()
    err = rel_max(got, ref)
    report(case, f"float64 max err / max = {err:.2e}")
    assert torch.allclose(got, ref, rtol=8e-3, atol=8e-3), err     # test_upsample2x_cat's bar: one bf16 rounding


# ------------------------------------------------------------------------------------------------ float32 mode
@gpu
@pytest.mark.parametrize("case", ["x3_linear_pg0", "x3_linear_pq"])
def test_gemm_x3_linear(ops, case):
    """cp_gemm_x3 Linear over M = B N rows: the pre-graph layer [taps | graph feature] 256 + 256 -> 256 with LeakyReLU, and
    an EdgeConv's [P|Q] GEMM 256 -> 512."""
    B = need_memory(case)
    g = gen(len(case))
    pg0 = case.endswith("pg0")
    K2, nout = (256, 256) if pg0 else (0, 512)
    a1 = randn(B, N, 256, g=g)
    a2 = randn(B, N, K2, g=g) if K2 else None
    w = randn(nout, 256 + K2, g=g) / (256 + K2) ** 0.5
    bias = randn(nout, g=g)
    ws = ops.pack_weight_split(w)

    def run(b0, b1):
        return (ops.gemm_x3_linear(a1[b0:b1], ws, nout, bias, pg0, 0.01, a2=None if a2 is None else a2[b0:b1]),)
    big = run(0, B)
    check_size(case, "a1", a1)
    if a2 is not None:
        check_size(case, "a2", a2)
    check_size(case, "out", big[0])
    check_slices(case, run, big)
    r = torch.tensor(boundary_rois(case), device="cuda")
    x = a1[r] if a2 is None else torch.cat([a1[r], a2[r]], -1)
    ref = x.double() @ w.double().t() + bias.double()
    if pg0:
        ref = lrelu64(ref, 0.01)
    err = rel_max(big[0][r], ref)
    report(case, f"float64 max err / max = {err:.2e}")
    assert err < 2e-5, err


@gpu
def test_gemm_x3_conv(ops):
    """cp_gemm_x3 3x3 convolution 512 -> 256 at 64 x 64 (up_net[2] in float32 mode) over a (B,64,64,512) fp32 map."""
    case = "x3_conv"
    B = need_memory(case)
    g = gen(4608)
    x = randn(B, 64, 64, 512, g=g)
    w = randn(256, 512, 3, 3, g=g) / 4608 ** 0.5
    bias = randn(256, g=g)
    ws = ops.pack_weight_split(w.permute(0, 2, 3, 1).reshape(256, 4608).contiguous())

    def run(b0, b1):
        return (ops.gemm_x3_conv(x[b0:b1], ws, 256, 3, 3, 1, 64, 64, bias, True, 0.0),)
    big = run(0, B)
    check_size(case, "x", x)
    check_size(case, "out", big[0])
    check_slices(case, run, big)
    r = torch.tensor(boundary_rois(case), device="cuda")
    ref = torch.relu(F.conv2d(x[r].permute(0, 3, 1, 2).double(), w.double(), bias.double(), padding=1)).permute(0, 2, 3, 1)
    err = rel_max(big[0][r], ref)
    report(case, f"float64 max err / max = {err:.2e}")
    assert err < 2e-5, err


@gpu
def test_edge_aggregate_staged_f32(ops, ycbv_plan):
    """cp_edge_aggregate_staged_f32 on the ycbv K = 20 plan with a graph per RoI: (B,N,512) fp32 -> (B,N,256)."""
    case = "agg_f32"
    B = need_memory(case)
    g = gen(2020)
    z = randn(B, N, 512, g=g)
    sel = torch.randint(0, G_YCBV, (B,), generator=g, device="cuda", dtype=torch.int32)

    def run(b0, b1):
        return (ops.edge_aggregate_staged(z[b0:b1], ycbv_plan, sel[b0:b1], 0.2),)
    big = run(0, B)
    check_size(case, "z", z)
    check_size(case, "out", big[0])
    check_slices(case, run, big)
    rois = boundary_rois(case)
    r, _, _ = rows_of(rois)
    R = len(rois)
    bi, ni = torch.arange(R, device="cuda").repeat_interleave(N), torch.arange(N, device="cuda").repeat(R)
    ref = agg_rows(z[r], ycbv_plan.idx_p[sel[r].long()].long(), bi, ni, 256, 0.2, False)
    assert torch.equal(big[0][r].reshape(-1, 256), ref), "aggregation must be bit-exact"
    report(case, "bit-exact")


@gpu
def test_sample_taps_f32(ops):
    """cp_sample_taps in float32 mode: 4 taps of a (B,65,65,64) patch map per keypoint, times the RoI mask -> (B,N,256)."""
    case = "taps_f32"
    B = need_memory(case)
    g = gen(256)
    patches = randn(B, 65, 65, 64, g=g)
    x_id = torch.randint(0, 32, (B, N), generator=g, device="cuda")
    y_id = torch.randint(0, 32, (B, N), generator=g, device="cuda")
    mask = (torch.rand(B, N, generator=g, device="cuda") > 0.2).float()

    def run(b0, b1):
        return (ops.sample_taps(patches[b0:b1], x_id[b0:b1], y_id[b0:b1], mask[b0:b1], 2),)
    big = run(0, B)
    for name, t in (("patches", patches), ("x_id", x_id), ("y_id", y_id), ("mask", mask), ("out", big[0])):
        check_size(case, name, t)
    check_slices(case, run, big)
    _, bi, ni = rows_of(boundary_rois(case))
    yy, xx = 2 * y_id[bi, ni], 2 * x_id[bi, ni]
    ref = torch.cat([patches[bi, yy + dy, xx + dx] for dy, dx in ((0, 0), (2, 0), (0, 2), (2, 2))], dim=-1) * mask[bi, ni, None]
    assert torch.equal(big[0][bi, ni], ref), "taps must be bit-exact"
    report(case, "bit-exact")
