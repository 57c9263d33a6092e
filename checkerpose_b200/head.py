"""Host-side orchestration of the GNN keypoint head on top of the C-ABI kernels.

This is the engine shared by the drop-in modules in ``checkerpose_b200/model``: weight preparation
(EdgeConv folding, bf16 tile packing, BN folding of the image branch) and the node-major forward of
the init head, one refine stage and the whole progressive head.  Two compute modes:

* ``torch.float32``  -- exact mode: fp32 tensors in HBM; every GEMM and every convolution of the image branch on the
  tensor cores with operands split into bf16 hi + lo (``cp_gemm_x3``: three tcgen05.mma per product, ~2^-16 relative),
  fp32 aggregation; matches the reference to ~1e-5 and decodes bit-exactly outside the 1e-4 logit band.
* ``torch.bfloat16`` -- product mode: the fused tcgen05 chain kernel (``cp_chain_fwd``), bf16 tensors in
  HBM, fp32 accumulation in TMEM.

The image branch (``up_net``, ``patch_generator``, ``seg_block``, ``conv1x1``) is dense convolution: in bf16 mode it
stays on cuDNN/cuBLAS through torch, as SURVEY.md section 8 marks it (library part of the path); in float32 mode it runs
on the implicit-GEMM form of ``cp_gemm_x3``.
"""
from __future__ import annotations

import contextlib

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops

_COMPUTE_DTYPE = torch.float32


def set_compute_dtype(dtype) -> None:
    """Select the arithmetic of the head: torch.float32 (validation) or torch.bfloat16 (product)."""
    global _COMPUTE_DTYPE
    if isinstance(dtype, str):
        dtype = {"fp32": torch.float32, "float32": torch.float32, "bf16": torch.bfloat16, "bfloat16": torch.bfloat16}[dtype]
    if dtype not in (torch.float32, torch.bfloat16):
        raise ValueError("compute dtype must be float32 or bfloat16")
    _COMPUTE_DTYPE = dtype


def get_compute_dtype():
    return _COMPUTE_DTYPE


# --------------------------------------------------------------------------------------------------
# bf16 widths.  The chain kernel takes widths that are multiples of 64 up to 512 (the patch-embedding width E of a refine
# stage a multiple of 16 up to 128).  Any other width runs padded: each node-major feature is stored with its channels
# rounded up to that granularity, the extra channels being exact zeros, and every weight gets zero rows for padded outputs,
# zero columns for padded inputs and zero bias.  A padded channel of a Linear is then 0 + 0 = 0, LeakyReLU(0) = 0, and it
# meets only zero weights downstream, so it adds exactly 0 to every real channel's sum.  An EdgeConv pads its convolution
# and BatchNorm before the fold, BatchNorm with gamma = beta = mean = 0 and var = 1: the folded scale and shift of a padded
# channel are 0, its [P|Q] columns are 0, and the aggregation lrelu(max_k P + Q) of zeros is 0.  Results handed back to
# the caller are sliced to the true width.
# --------------------------------------------------------------------------------------------------
MAX_BF16_WIDTH = 512
MAX_BF16_EMBED = 128


def pad64(c: int) -> int:
    return (c + 63) // 64 * 64


def pad16(c: int) -> int:
    return (c + 15) // 16 * 16


def _pad_segments(t, dim, segs, value=0.0):
    """Zero-pad ``t`` along ``dim`` segment by segment: ``segs`` = ((true, padded), ...) laid end to end."""
    if all(a == b for a, b in segs):
        return t
    parts, o = [], 0
    for a, b in segs:
        x = t.narrow(dim, o, a)
        if b > a:
            shape = list(x.shape)
            shape[dim] = b - a
            x = torch.cat([x, torch.full(shape, value, dtype=t.dtype, device=t.device)], dim)
        parts.append(x)
        o += a
    return torch.cat(parts, dim)


def pad_linear_weight(weight, bias, rows, cols):
    """(nout, kin) weight and (nout) bias zero-padded: ``rows`` / ``cols`` = ((true, padded), ...) segments."""
    w = weight.detach().reshape(weight.shape[0], -1).float()
    w = _pad_segments(_pad_segments(w, 0, rows), 1, cols)
    b = None if bias is None else _pad_segments(bias.detach().float(), 0, rows)
    return w, b


def pad_edgeconv(w, gamma, beta, mean, var):
    """EdgeConv convolution (C', 2C[, 1, 1]) and BatchNorm parameters padded before the fold: C -> pad64(C) on both halves of
    the [x_j - x_i | x_i] input, C' -> pad64(C') with gamma = beta = mean = 0 and var = 1 (folded scale and shift 0)."""
    co, c = w.shape[0], w.shape[1] // 2
    rows, half = ((co, pad64(co)),), (c, pad64(c))
    w = _pad_segments(_pad_segments(w.reshape(co, 2 * c).float(), 0, rows), 1, (half, half))
    gamma, beta, mean = (_pad_segments(t.float(), 0, rows) for t in (gamma, beta, mean))
    return w, gamma, beta, mean, _pad_segments(var.float(), 0, rows, 1.0)


def _pad_to(x, width):
    """Node-major x (B,N,c) with its channels zero-padded to ``width`` (no copy when it already has them)."""
    return x if x.shape[-1] == width else F.pad(x, (0, width - x.shape[-1]))


def check_bf16_width(what: str, c: int, limit: int = MAX_BF16_WIDTH) -> None:
    if c > limit:
        raise RuntimeError(f"bf16 mode runs {what} up to {limit} channels (got {c}); use float32 mode for wider heads")


# --------------------------------------------------------------------------------------------------
# prepared weights (derived from the module parameters; never stored in the state_dict)
# --------------------------------------------------------------------------------------------------
class PreparedLinear:
    """bf16 mode: ``packed`` = bf16 tile image for the chain / EdgeConv kernels.  float32 mode: ``split`` = the
    (hi, lo) bf16 tile images of the split-precision tensor-core GEMM (cp_gemm_x3); layers whose K is not a multiple
    of 64 keep the SIMT GEMM.  ``nout`` / ``kin`` are the widths of the (possibly padded) weight."""

    def __init__(self, weight, bias, want_packed):
        self.w = weight.detach().reshape(weight.shape[0], -1).contiguous().float()
        self.b = None if bias is None else bias.detach().contiguous().float()
        self.nout, self.kin = self.w.shape
        self.packed = ops.pack_weight(self.w) if (want_packed and self.kin % 64 == 0) else None
        self.split = ops.pack_weight_split(self.w) if (not want_packed and self.kin % 64 == 0 and self.w.is_cuda) else None


def linear32(x, prep: "PreparedLinear", act=False, slope=0.0, a2=None):
    """float32 mode: y = act([x|a2] @ W.T + b) -- split-bf16 x3 on tcgen05 when the shape allows, else SIMT FFMA."""
    k2 = 0 if a2 is None else a2.shape[-1]
    if prep.split is not None and x.shape[-1] % 64 == 0 and k2 % 64 == 0:
        return ops.gemm_x3_linear(x, prep.split, prep.nout, prep.b, act, slope, a2=a2)
    return ops.linear_f32(x, prep.w, prep.b, act, slope, a2=a2)


class PreparedEdgeConv(PreparedLinear):
    """StaticGraph_module weights folded to the factored form [P|Q] (see cp_fold_edgeconv)."""

    def __init__(self, sg_module, want_packed, pad=False):
        conv, bn, act = sg_module.conv[0], sg_module.conv[1], sg_module.conv[2]
        w, gamma, beta = conv.weight.detach(), bn.weight.detach(), bn.bias.detach()
        mean, var = bn.running_mean.detach(), bn.running_var.detach()
        if pad:
            w, gamma, beta, mean, var = pad_edgeconv(w, gamma, beta, mean, var)
        wf, bf = ops.fold_edgeconv(w, gamma, beta, mean, var, bn.eps)
        super().__init__(wf, bf, want_packed)
        self.C, self.Co = wf.shape[1], wf.shape[0] // 2
        self.slope = float(act.negative_slope)
        if self.slope < 0.0:
            # lrelu(max_k P_j + Q_i) == max_k lrelu(P_j + Q_i) needs an increasing activation
            raise RuntimeError("the factored EdgeConv kernels need a LeakyReLU with negative_slope >= 0 "
                               f"(got {self.slope}): the max over neighbours must commute with the activation")


def _ver(t: torch.Tensor) -> int:
    """Version counter of a tensor.  Inference tensors (created under ``torch.inference_mode()``) do not track one and
    raise when ``_version`` is read; they cannot be modified in place outside inference mode either, so a constant is a
    valid cache key for them (a replaced tensor has another ``data_ptr`` / identity)."""
    return -1 if t.is_inference() else t._version


def _param_fingerprint(module: nn.Module):
    return tuple((t.data_ptr(), _ver(t), t.device, t.dtype) for t in list(module.parameters()) + list(module.buffers()))


class PrepCache:
    """Lazily (re)built prepared weights.  The cache lives ON the owning module (so it dies with it -- a
    global table keyed by ``id()`` / ``data_ptr()`` would hand a new module the stale weights of a freed
    one whose addresses were recycled) and is invalidated when parameters change version or move."""

    _ATTR = "_cp_prepared"

    def get(self, owner: nn.Module, key, builder):
        store = owner.__dict__.get(self._ATTR)
        if store is None:
            store = {}
            owner.__dict__[self._ATTR] = store
        fp = _param_fingerprint(owner)
        hit = store.get(key)
        if hit is None or hit[0] != fp:
            hit = (fp, builder())
            store[key] = hit
        return hit[1]


_PREP = PrepCache()


def prepared_edgeconv(sg_module, dtype) -> PreparedEdgeConv:
    """bf16 mode: input and output widths padded to multiples of 64 (unchanged when they are)."""
    want = dtype == torch.bfloat16
    co, c2 = sg_module.conv[0].weight.shape[:2]
    pad = want and (co % 64 != 0 or (c2 // 2) % 64 != 0)
    return _PREP.get(sg_module, ("ec", want, pad), lambda: PreparedEdgeConv(sg_module, want, pad))


def prepared_linear(lin: nn.Module, dtype, rows=None, cols=None) -> PreparedLinear:
    """``rows`` / ``cols``: ((true, padded), ...) segments the bf16 weight is zero-padded to (see pad_linear_weight)."""
    want = dtype == torch.bfloat16
    rows = ((lin.weight.shape[0],) * 2,) if rows is None else tuple(rows)
    cols = ((lin.weight.shape[1],) * 2,) if cols is None else tuple(cols)
    if all(a == b for a, b in rows + cols):
        return _PREP.get(lin, ("lin", want), lambda: PreparedLinear(lin.weight, lin.bias, want))
    return _PREP.get(lin, ("lin", want, rows, cols), lambda: PreparedLinear(*pad_linear_weight(lin.weight, lin.bias, rows, cols), want))


def _padded_linear(lin: nn.Module, kin_stored: int, last: bool = False) -> PreparedLinear:
    """bf16 Linear reading a stored input of ``kin_stored`` (>= in_features) channels; its output padded to a multiple of
    64 unless it is the ``last`` layer (an f32 result with n_valid columns)."""
    nout, kin = lin.weight.shape
    check_bf16_width("a Linear layer", max(kin, nout))
    return prepared_linear(lin, torch.bfloat16, rows=((nout, nout if last else pad64(nout)),), cols=((kin, kin_stored),))


class GraphTable:
    """int32 copy of a module's kNN index table: (G,N,K); G=1 for the single-object nets.  Cached as an
    attribute of the index tensor itself (never in a table keyed by a recyclable address)."""

    @classmethod
    def get(cls, knn_idx: torch.Tensor, device) -> torch.Tensor:
        device = torch.device(device)
        hit = getattr(knn_idx, "_cp_idx32", None)
        if hit is None or hit[0] != _ver(knn_idx) or hit[1].device != device:
            hit = (_ver(knn_idx), knn_idx.to(device=device, dtype=torch.int32).contiguous())
            knn_idx._cp_idx32 = hit
        return hit[1]


def _graph_tensor(knn_src, device):
    return knn_src.get(device) if hasattr(knn_src, "get") else knn_src


def graph_select(knn_idx, obj_ids, batch: int, device):
    """-> (idx32 (G,N,K) in keypoint numbering, graph_sel int32 (B) or None).  LM nets index with 1-based ids
    (pipeline_lm.py:56-57)."""
    idx32 = GraphTable.get(_graph_tensor(knn_idx, device), device)
    return idx32, _graph_sel(idx32.shape[0], obj_ids, batch, device)


def _graph_sel(G, obj_ids, batch, device):
    if obj_ids is not None:
        # 1-based object ids -> 0-based graph selector; ids outside [1, G] trap on the device (the reference's
        # ``self.knn_idx[obj_ids-1]`` raises a device-side index assert for them)
        return ops.graph_sel(obj_ids.to(device=device), G)
    if G == 1:
        return None
    if G != batch:
        raise RuntimeError(f"knn_idx has {G} graphs for a batch of {batch}")
    return torch.arange(batch, dtype=torch.int32, device=device)


class GraphCtx:
    """What the kernels need to know about a module's static graph for one batch: the plan (keypoint renumbering,
    plan-order neighbour table, staging lists) and the per-RoI graph selector."""

    __slots__ = ("plan", "sel")

    def __init__(self, plan, sel):
        self.plan, self.sel = plan, sel

    def to_plan(self, x_nm):
        """(B,N,...) keypoint order -> plan order."""
        return x_nm if self.plan.identity else ops.permute_rows(x_nm, self.plan.perm, self.sel, False)

    def to_keypoints(self, x_nm):
        """(B,N,...) plan order -> keypoint order."""
        return x_nm if self.plan.identity else ops.permute_rows(x_nm, self.plan.perm, self.sel, True)


def graph_ctx(knn_src, obj_ids, batch: int, device) -> GraphCtx:
    """Plan of a module's graph (built once, cached on the graph object) + selector for this batch."""
    device = torch.device(device)
    t = _graph_tensor(knn_src, device)
    hit = getattr(t, "_cp_plan", None)
    if hit is None or hit[0] != _ver(t) or hit[1].perm.device != device:
        xyz = getattr(knn_src, "p3d_normed", None)
        hit = (_ver(t), ops.GraphPlan(GraphTable.get(t, device), xyz))
        t._cp_plan = hit
    plan = hit[1]
    return GraphCtx(plan, _graph_sel(plan.G, obj_ids, batch, device))


def _first_cuda_device(args, kwargs):
    for a in list(args) + list(kwargs.values()):
        if isinstance(a, torch.Tensor) and a.is_cuda:
            return a.device
        if isinstance(a, (list, tuple)):
            for t in a:
                if isinstance(t, torch.Tensor) and t.is_cuda:
                    return t.device
    return None


class DeviceScopedModule(nn.Module):
    """nn.Module whose call runs with the CUDA device of its first tensor argument current: the kernels launch on the
    current device's current stream (ops._need_cuda), so a net moved to ``cuda:1`` works without ``torch.cuda.set_device``."""

    def __call__(self, *args, **kwargs):
        dev = _first_cuda_device(args, kwargs)
        if dev is None or dev.index == torch.cuda.current_device():
            return super().__call__(*args, **kwargs)
        with torch.cuda.device(dev):
            return super().__call__(*args, **kwargs)


def _require_eval(module):
    if module.training:
        raise RuntimeError("checkerpose_b200 kernels fold BatchNorm running statistics and are inference-only: "
                           "call .eval() (training-mode BN over B*N*K is out of scope)")


# --------------------------------------------------------------------------------------------------
# EdgeConv (K2).  Every node-major tensor below is in PLAN order (GraphCtx.to_plan / to_keypoints convert).
# --------------------------------------------------------------------------------------------------
def _agg_gemm(z, ctx: GraphCtx, agg_slope, layer, out, out_mode, n_valid=0, a_out=None):
    """A = EdgeConv aggregation of the [P|Q] table z; out = layer(A).  Staged warp-specialised kernel when the
    graph plan and the widths fit it (C' in {64,128,256}, out <= 512 columns), else the unstaged chain kernel with direct
    global gathers."""
    if ctx.plan.staged and z.shape[-1] // 2 in (64, 128, 256) and layer.nout <= 512:
        return ops.edgeconv_fwd(z=z, plan=ctx.plan, graph_sel=ctx.sel, agg_slope=agg_slope, layer=layer, out=out,
                                out_mode=out_mode, n_valid=n_valid, a_out=a_out)
    return ops.chain_fwd(prologue=ops.PRO_AGG, B=z.shape[0], N=z.shape[1], z=z, idx32=ctx.plan.idx_p, graph_sel=ctx.sel,
                         agg_slope=agg_slope, a_out=a_out, layers=[layer], out=out, out_mode=out_mode, n_valid=n_valid)


def edgeconv_node_major(sg_module, x_nm, ctx: GraphCtx, dtype):
    """x_nm (B,N,C) of ``dtype`` -> (B,N,Co).  StaticGraph_module.forward (pipeline.py:55-59), one layer on its own."""
    _require_eval(sg_module)
    if dtype == torch.bfloat16:
        co, c2 = sg_module.conv[0].weight.shape[:2]
        check_bf16_width("an EdgeConv", max(co, c2 // 2))
    prep = prepared_edgeconv(sg_module, dtype)
    B, N, _ = x_nm.shape
    if dtype == torch.float32:
        z = linear32(x_nm, prep)
        if ctx.plan.struct is not None and ctx.plan.max_unique <= ops.PLAN_UMAX and prep.Co % 32 == 0:
            return ops.edge_aggregate_staged(z, ctx.plan, ctx.sel, prep.slope)     # rows staged in shared memory per tile
        return ops.edge_aggregate(z, ctx.plan.idx_p, ctx.sel, prep.slope)
    # bf16: widths padded to multiples of 64; the result keeps the padded channels (zeros)
    z = torch.empty((B, N, 2 * prep.Co), dtype=torch.bfloat16, device=x_nm.device)
    ops.chain_fwd(prologue=ops.PRO_LOAD, B=B, N=N, src=_pad_to(x_nm, prep.C),
                  layers=[ops.chain_layer(prep.packed, prep.b, prep.C, 2 * prep.Co, False, 0.0)], out=z, out_mode=ops.OUT_BF16)
    return ops.edge_aggregate(z, ctx.plan.idx_p, ctx.sel, prep.slope)


# --------------------------------------------------------------------------------------------------
# init head (InitNet_GNN.forward after the backbone, init.py:112-122)
# --------------------------------------------------------------------------------------------------
def init_head_node_major(init_net, feat_last, obj_ids, dtype):
    """-> logits (B,N,>=7) f32, graph feature (B,N,64) of ``dtype`` (both in plan order), GraphCtx (None without
    graph modules)."""
    _require_eval(init_net)
    B = feat_last.shape[0]
    N = init_net.npoint
    dev = feat_last.device
    bias0 = None
    if dtype == torch.bfloat16 and _IMAGE_BRANCH == "cudnn":
        conv = _bf16_module(init_net.conv1x1)
        x0, bias0 = conv(feat_last.to(torch.bfloat16), defer_last_bias=True)   # bias applied by the layout change below
    else:
        x0 = image_block(init_net.conv1x1, feat_last, dtype)                   # 1x1 conv = split-precision GEMM, NHWC result
    blocks = list(init_net.pre_query_block)
    mlp = prepared_linear(init_net.mlp, dtype)
    nbits = mlp.nout
    ctx = graph_ctx(blocks[0]._knn, obj_ids, B, dev) if blocks else None
    # == out.view(-1, N, 64): channel = 8x8 cell (init.py:114)
    hw = x0.shape[2] * x0.shape[3]
    if (dtype == torch.bfloat16 and x0.is_contiguous(memory_format=torch.channels_last) and not x0.is_contiguous()
            and hw % 64 == 0 and N % 64 == 0):
        # (B,hw,N) -> (B,N,hw) + conv bias + keypoint -> plan order in one tiled pass
        row_map = None if ctx is None or ctx.plan.identity else ctx.plan.perm_inv
        x = ops.transpose_scatter(x0.permute(0, 2, 3, 1).reshape(B, hw, N), bias0, row_map, None if ctx is None else ctx.sel)
    else:
        if bias0 is not None:
            x0 = x0 + bias0.to(x0.dtype).view(1, -1, 1, 1)
        if x0.permute(0, 2, 3, 1).is_contiguous():      # NHWC storage (B,hw,N) -> (B,N,hw) with the tiled transpose
            x = ops.to_node_major(x0.permute(0, 2, 3, 1).reshape(B, hw, N), x0.dtype)
        else:
            x = x0.contiguous().view(B, N, hw)
        if ctx is not None:
            x = ctx.to_plan(x)
    if dtype == torch.float32:
        for blk in blocks:
            x = edgeconv_node_major(blk, x, ctx, dtype)
        logits = linear32(x, mlp)
        return logits, x, ctx
    # bf16: LOAD->[W_0] ; AGG->[W_j] ... ; AGG(+store feature)->[mlp]
    logits = torch.empty((B, N, 16), dtype=torch.float32, device=dev)
    mlp_layer = ops.chain_layer(mlp.packed, mlp.b, 64, nbits, False, 0.0)
    if not blocks:
        ops.chain_fwd(prologue=ops.PRO_LOAD, B=B, N=N, src=x, layers=[mlp_layer], out=logits, out_mode=ops.OUT_F32, n_valid=nbits)
        return logits, x, ctx
    preps = [prepared_edgeconv(b, dtype) for b in blocks]
    for b in blocks:
        _require_eval(b)
    z = torch.empty((B, N, 2 * preps[0].Co), dtype=torch.bfloat16, device=dev)
    ops.chain_fwd(prologue=ops.PRO_LOAD, B=B, N=N, src=x,
                  layers=[ops.chain_layer(preps[0].packed, preps[0].b, preps[0].C, 2 * preps[0].Co, False, 0.0)],
                  out=z, out_mode=ops.OUT_BF16)
    for j in range(1, len(blocks)):
        z2 = torch.empty((B, N, 2 * preps[j].Co), dtype=torch.bfloat16, device=dev)
        _agg_gemm(z, ctx, preps[j - 1].slope, ops.chain_layer(preps[j].packed, preps[j].b, preps[j].C, 2 * preps[j].Co, False, 0.0),
                  z2, ops.OUT_BF16)
        z = z2
    gfeat = torch.empty((B, N, preps[-1].Co), dtype=torch.bfloat16, device=dev)
    _agg_gemm(z, ctx, preps[-1].slope, mlp_layer, logits, ops.OUT_F32, n_valid=nbits, a_out=gfeat)
    return logits, gfeat, ctx


# --------------------------------------------------------------------------------------------------
# image branch: one BN-folded description of a conv stack, three executors built from it
# --------------------------------------------------------------------------------------------------
def image_layers(module):
    """The layers of an image-branch module (up_net block, patch_generator, seg_block, conv1x1: an nn.Sequential or one
    layer), walked once, as tuples ``(kind, w, b, m, relu)``.  A convolution (kind "conv" / "convT") carries its fp32 weight
    ``w`` in the module's own layout and its fp32 bias ``b`` (or None), with a following BatchNorm2d folded in on the output
    channels (axis 0 of a Conv2d weight, axis 1 of a ConvTranspose2d weight), the module ``m`` itself (stride, padding, ...)
    and whether a following ReLU is fused.  "relu", "lrelu" and "up" (UpsamplingBilinear2d(scale_factor=2)) entries carry
    only ``m``.  Every executor builds from this list, so all of them run bit-identical folded weights."""
    mods = list(module) if isinstance(module, nn.Sequential) else [module]
    layers = []
    i = 0
    while i < len(mods):
        m = mods[i]
        if isinstance(m, (nn.Conv2d, nn.ConvTranspose2d)):
            tr = isinstance(m, nn.ConvTranspose2d)
            w = m.weight.detach().float()
            b = None if m.bias is None else m.bias.detach().float()
            if i + 1 < len(mods) and isinstance(mods[i + 1], nn.BatchNorm2d):
                bn = mods[i + 1]
                sc = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
                sh = bn.bias.detach().float() - sc * bn.running_mean.detach().float()
                w = w * (sc.view(1, -1, 1, 1) if tr else sc.view(-1, 1, 1, 1))
                b = sh if b is None else b * sc + sh
                i += 1
            relu = i + 1 < len(mods) and isinstance(mods[i + 1], nn.ReLU)
            if relu:
                i += 1
            layers.append(("convT" if tr else "conv", w, b, m, relu))
        elif isinstance(m, nn.ReLU):
            layers.append(("relu", None, None, m, False))
        elif isinstance(m, nn.LeakyReLU):
            layers.append(("lrelu", None, None, m, False))
        elif isinstance(m, nn.UpsamplingBilinear2d):
            if float(m.scale_factor) != 2.0:
                raise RuntimeError("image branch: only UpsamplingBilinear2d(scale_factor=2) is supported")
            layers.append(("up", None, None, m, False))
        else:
            raise RuntimeError(f"unsupported layer in image branch: {type(m).__name__}")
        i += 1
    return layers


def _gemm_layers(module, pack, mode):
    """image_layers(module) for our implicit-GEMM kernels: each convolution as (kind, pack(W rows in (ky, kx, c) order, Cin
    zero-padded to the kernels' 64-channel K chunks), b, (cout, kh, kw, pad, cin_pad), relu).  They take Conv2d stride 1 and
    ConvTranspose2d stride 2 / output_padding 1 with square padding, no dilation or groups, and ReLU but not LeakyReLU;
    ``mode`` names the branch in the error raised for anything else."""
    layers = []
    for kind, w, b, m, relu in image_layers(module):
        if kind in ("relu", "up"):
            layers.append((kind, None, None, None, False))
            continue
        tr = kind == "convT"
        if kind == "lrelu" or not (m.groups == 1 and tuple(m.dilation) == (1, 1) and m.padding[0] == m.padding[1] and
                                   tuple(m.stride) == ((2, 2) if tr else (1, 1)) and (not tr or tuple(m.output_padding) == (1, 1))):
            raise RuntimeError(f"{mode} image branch: unsupported layer {m}")
        kh, kw = m.kernel_size
        cin, cout = (w.shape[0], w.shape[1]) if tr else (w.shape[1], w.shape[0])
        wk = w.permute(1, 2, 3, 0) if tr else w.permute(0, 2, 3, 1)        # (cout, kh, kw, cin)
        cin_pad = (cin + 63) // 64 * 64
        if cin_pad != cin:
            wk = F.pad(wk, (0, cin_pad - cin))
        layers.append((kind, pack(wk.reshape(cout, kh * kw * cin_pad).contiguous()), None if b is None else b.contiguous(),
                       (cout, kh, kw, int(m.padding[0]), cin_pad), relu))
    return layers


def _nhwc(x, dtype):
    """NCHW (any strides) -> contiguous (B,H,W,C) of ``dtype``: a view when x already is one, else one launch of
    cp_transpose_cn_to_nc (the tiled transpose for the bf16 HRNet maps)."""
    v = x.permute(0, 2, 3, 1)
    if v.is_contiguous() and v.dtype == dtype:
        return v
    B, Cc, H, W = x.shape
    return ops.to_node_major(x.contiguous().view(B, Cc, H * W), dtype).view(B, H, W, Cc)


def _pad_channels(y, cin_pad):
    """Zero channels of an NHWC map up to the implicit-GEMM kernels' 64-channel granularity."""
    return y if y.shape[-1] == cin_pad else F.pad(y, (0, cin_pad - y.shape[-1]))


def _gather_conv(conv, y, kind, ws, b, geom, relu):
    """One convolution of a _gemm_layers entry on a gather kernel (ops.gemm_x3_conv / ops.conv_bf16) over the contiguous NHWC
    map y; stride 1 for "conv", stride 2 with output_padding 1 for "convT"."""
    cout, kh, kw, pad, cin_pad = geom
    y = _pad_channels(y, cin_pad)
    H, W = y.shape[1], y.shape[2]
    if kind == "conv":
        Ho, Wo = H + 2 * pad - kh + 1, W + 2 * pad - kw + 1
    else:
        Ho, Wo = (H - 1) * 2 - 2 * pad + kh + 1, (W - 1) * 2 - 2 * pad + kw + 1
    return conv(y, ws, cout, kh, kw, pad, Ho, Wo, b, relu, 0.0, transposed=(kind == "convT"))


class _FoldedSeq:
    """bf16, channels_last, BN-folded functional copy of a conv stack (up_net block / single conv).
    Convolutions run on cuDNN (library part of the path); the bilinear x2 upsampling of the concatenated
    skip connection runs on cp_upsample2x_cat_nhwc (one pass, no materialised concat)."""

    _fused_relu_ok = None   # torch.cudnn_convolution_relu availability, probed on first use

    def __init__(self, module):
        self.ops = []
        self.bias_f32 = {}     # op index -> f32 bias (the bf16 copy in ops is what cuDNN's fused conv+bias+ReLU takes)
        for kind, w, b, m, relu in image_layers(module):
            if w is not None:
                self.bias_f32[len(self.ops)] = None if b is None else b.contiguous()
                w = w.to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
                b = None if b is None else b.to(torch.bfloat16)
            self.ops.append((kind, w, b, m, relu))

    @classmethod
    def _conv_relu(cls, x, w, b, m):
        if cls._fused_relu_ok is not False and b is not None and m.groups == 1:
            try:
                y = torch.cudnn_convolution_relu(x, w, b, m.stride, m.padding, m.dilation, m.groups)
                cls._fused_relu_ok = True
                return y
            except (RuntimeError, AttributeError):
                cls._fused_relu_ok = False
        return torch.relu_(F.conv2d(x, w, b, stride=m.stride, padding=m.padding, dilation=m.dilation, groups=m.groups))

    @staticmethod
    def _bias_act(y, bias_f32, relu):
        """[relu](y + bias) in place on a channels-last conv output: one pass of cp_bias_add_rows_bf16 instead of torch's
        broadcast add (+ clamp)."""
        v = y.permute(0, 2, 3, 1)
        if bias_f32 is not None and v.is_contiguous() and v.shape[-1] % 8 == 0:
            ops.bias_add_rows_(v, bias_f32, relu)
            return y
        if bias_f32 is not None:
            y = y + bias_f32.to(y.dtype).view(1, -1, 1, 1)
        return torch.relu_(y) if relu else y

    def __call__(self, x, skip=None, defer_last_bias=False):
        """defer_last_bias: return (y, bias) with the last convolution's bias NOT applied (its consumer fuses it)."""
        start = 0
        last = len(self.ops) - 1
        if self.ops[0][0] == "up":
            a = _nhwc(x, torch.bfloat16).permute(0, 3, 1, 2)
            s = None if skip is None else _nhwc(skip, torch.bfloat16).permute(0, 3, 1, 2)
            x = ops.upsample2x_cat(a, s)
            start = 1
        else:
            if skip is not None:
                x = torch.cat([x, skip], dim=1)
            x = _nhwc(x, torch.bfloat16).permute(0, 3, 1, 2)
        for oi, (kind, w, b, m, relu) in enumerate(self.ops[start:], start):
            if kind == "conv":
                if relu and b is not None:
                    x = self._conv_relu(x, w, b, m)
                else:
                    x = F.conv2d(x, w, None, stride=m.stride, padding=m.padding, dilation=m.dilation, groups=m.groups)
                    if defer_last_bias and oi == last and not relu:
                        return x, self.bias_f32[oi]
                    x = self._bias_act(x, self.bias_f32[oi], relu)
            elif kind == "convT":
                x = F.conv_transpose2d(x, w, None, stride=m.stride, padding=m.padding, output_padding=m.output_padding)
                x = self._bias_act(x, self.bias_f32[oi], relu)
            elif kind == "relu":
                x = torch.relu_(x)
            elif kind == "lrelu":
                x = F.leaky_relu(x, m.negative_slope)
            else:
                x = ops.upsample2x_cat(_nhwc(x, torch.bfloat16).permute(0, 3, 1, 2), None)
        return (x, None) if defer_last_bias else x


class _X3ConvSeq:
    """The float32 image branch: every convolution of a conv stack one launch of the split-precision implicit GEMM cp_gemm_x3
    over fp32 NHWC maps, bias + ReLU in its epilogue; the bilinear x2 upsampling of the concatenated skip connection runs on
    cp_upsample2x_cat_nhwc.  NCHW in, NCHW (channels_last strides) out."""

    def __init__(self, module):
        self.ops = _gemm_layers(module, ops.pack_weight_split, "float32")

    def __call__(self, x, skip=None):
        start = 0
        if self.ops[0][0] == "up":
            a = _nhwc(x, torch.float32).permute(0, 3, 1, 2)
            s = None if skip is None else _nhwc(skip, torch.float32).permute(0, 3, 1, 2)
            y = ops.upsample2x_cat(a, s).permute(0, 2, 3, 1)         # (B,2H,2W,Ca+Cb) contiguous
            start = 1
        else:
            if skip is not None:
                x = torch.cat([x, skip], dim=1)
            y = _nhwc(x, torch.float32)
        for kind, ws, b, geom, relu in self.ops[start:]:
            if kind in ("conv", "convT"):
                y = _gather_conv(ops.gemm_x3_conv, y, kind, ws, b, geom, relu)
            elif kind == "relu":
                y = torch.relu_(y)
            else:
                y = ops.upsample2x_cat(y.permute(0, 3, 1, 2), None).permute(0, 2, 3, 1)
        return y.permute(0, 3, 1, 2)


class _SlabConvSeq:
    """The bf16 image branch on cp_conv_slab: every map of a block lives in a BORDERED NHWC buffer (B, H+1, W+1, C) -- a zero
    last row and last column per image, which over the flat pixel index are all four borders at once -- so that a kernel tap is
    a row shift of one TMA-loaded activation slab (csrc/conv_slab_tcgen05.cu).  The x2 upsampling of the concatenated skip
    connection writes straight into a bordered buffer (cp_upsample2x_cat_nhwc_to), 3x3 / 1x1 convolutions map buffer to buffer (their epilogue rewrites the border as zeros),
    the transposed convolution of the first block runs as its four output parities, and patch_generator (2x2, padding 1)
    produces exactly the stored grid as a contiguous (B, H+1, W+1, E) map.  The NCHW view handed back to the caller is the interior of the
    buffer and remembers it (``_cp_padded``): the next block / patch_generator / seg_block pick the buffer up again
    without a copy.  Shapes the slab kernel does not take (more than 256 output channels: conv1x1 of the init head) fall
    back to the gather kernel cp_conv_bf16."""

    def __init__(self, module):
        self.ops = _gemm_layers(module, ops.pack_weight, "bf16")

    @staticmethod
    def _view(buf):
        y = buf[:, :-1, :-1, :].permute(0, 3, 1, 2)
        y._cp_padded = buf
        return y

    @staticmethod
    def _cl(x):
        """(B,C,H,W) -> a bf16 view / copy with channel stride 1 (what the upsampling kernel reads)."""
        if x.dtype == torch.bfloat16 and x.stride(1) == 1 and all(st % 8 == 0 for st in (x.stride(0), x.stride(2), x.stride(3))):
            return x
        return _nhwc(x, torch.bfloat16).permute(0, 3, 1, 2)

    def __call__(self, x, skip=None, seg=None):
        """``seg`` = (weight (n, C), bias (n,)) f32 of a 1x1 convolution to fuse into this block's LAST convolution: the
        result gains the attribute ``_cp_seg`` = its (B, n, H, W) f32 output (None when the shapes do not allow the fusion)."""
        kinds = self.ops
        start = 0
        seg_out = None
        buf = None          # zero-bordered (B,H+2,W+2,C) map, or None while y (plain NHWC) holds the current map
        y = None
        if kinds[0][0] == "up":
            buf = ops.upsample2x_cat_padded(self._cl(x), None if skip is None else self._cl(skip))
            start = 1
        elif kinds[0][0] == "convT" and kinds[0][3][1:4] == (3, 3, 1) and kinds[0][3][0] <= 256:
            _, ws, b, (cout, kh, kw, pad, cin_pad), relu = kinds[0]
            if skip is not None:
                x = torch.cat([x, skip], dim=1)
            buf = ops.convT_slab(_pad_channels(_nhwc(x, torch.bfloat16), cin_pad), ws, cout, b, relu, 0.0)
            start = 1
        else:
            buf = getattr(x, "_cp_padded", None) if skip is None else None
            if buf is None:
                if skip is not None:
                    x = torch.cat([x, skip], dim=1)
                y = _nhwc(x, torch.bfloat16)
        for oi in range(start, len(kinds)):
            kind, ws, b, geom, relu = kinds[oi]
            if kind == "relu":
                cur = buf if buf is not None else y
                torch.relu_(cur)
                continue
            if kind == "up":
                src = self._view(buf) if buf is not None else y.permute(0, 3, 1, 2)
                buf, y = ops.upsample2x_cat_padded(src, None), None
                continue
            cout, kh, kw, pad, cin_pad = geom
            same = kind == "conv" and kh == kw and kh in (1, 3) and pad == kh // 2
            full = kind == "conv" and kh == kw == 2 and pad == 1
            if cout <= 256 and (same or full):
                if buf is None:
                    buf, y = ops.to_bordered(y), None
                buf = _pad_channels(buf, cin_pad)
                if same:
                    if seg is not None and oi == len(kinds) - 1 and seg[0].shape[1] == cout:
                        buf, seg_out = ops.conv_slab_same(buf, ws, cout, kh, kw, b, relu, 0.0, seg=seg)
                    else:
                        buf = ops.conv_slab_same(buf, ws, cout, kh, kw, b, relu, 0.0)
                else:
                    y, buf = ops.conv_slab_full(buf, ws, cout, kh, kw, b, relu, 0.0), None
                continue
            # gather kernel on a contiguous map
            if buf is not None:
                y, buf = buf[:, :-1, :-1, :].contiguous(), None
            y = _gather_conv(ops.conv_bf16, y, kind, ws, b, geom, relu)
        res = self._view(buf) if buf is not None else y.permute(0, 3, 1, 2)
        res._cp_seg = seg_out
        return res


def _x3_module(module):
    _require_eval(module)
    return _PREP.get(module, ("x3seq",), lambda: _X3ConvSeq(module))


def _tc_module(module):
    _require_eval(module)
    return _PREP.get(module, ("tcseq",), lambda: _SlabConvSeq(module))


_IMAGE_BRANCH = "tcgen05"


def set_image_branch(kind: str) -> None:
    """bf16 mode only: "tcgen05" (default) = the image branch on our slab convolutions (cp_conv_slab; cp_conv_bf16 for conv1x1:
    no library kernel anywhere in the head), "cudnn" = the library convolutions through torch (SURVEY 8a marks them as the
    library part of the path; kept as the A/B arm).  Measured end to end (DESIGN.md section 8): within about 1 % of each other
    inside the power-capped step (14.55 vs 14.46 ms, 13.87 vs 13.87 ms on two boxes), with our kernels ahead on every
    convolution in isolation.  The float32 mode never uses a library kernel."""
    global _IMAGE_BRANCH
    if kind not in ("tcgen05", "cudnn"):
        raise ValueError("image branch must be 'tcgen05' or 'cudnn'")
    _IMAGE_BRANCH = kind


def get_image_branch() -> str:
    return _IMAGE_BRANCH


def _bf16_module(module):
    _require_eval(module)
    return _PREP.get(module, ("bf16seq",), lambda: _FoldedSeq(module))


_IMG_REUSE = None   # measurement aid, see reuse_image_branch()


@contextlib.contextmanager
def reuse_image_branch():
    """bench.py's "GNN-only" leg (SURVEY.md 8d asks for the GNN kernels and the whole head separately): inside this
    context the outputs of the library convolutions of the image branch (up_net, patch_generator, seg_block) are
    computed once per module and then reused, so a step of a FIXED input batch runs only the GNN path.  Never active
    in the product path or in the headline numbers."""
    global _IMG_REUSE
    _IMG_REUSE = {}
    try:
        yield
    finally:
        _IMG_REUSE = None


def _seg_weights(seg_module):
    """(weight (n, C) f32, bias (n,) f32) of a 1x1 seg_block that the slab convolution can fuse, else None."""
    m = seg_module
    if not (isinstance(m, nn.Conv2d) and m.kernel_size == (1, 1) and m.stride == (1, 1) and m.padding == (0, 0) and m.groups == 1
            and m.bias is not None and m.out_channels <= 4):
        return None
    return _PREP.get(m, ("segw",), lambda: (m.weight.detach().float().reshape(m.out_channels, -1).contiguous(), m.bias.detach().float().contiguous()))


def image_block(module, x, dtype, skip=None, seg_module=None):
    """Run an image-branch block (up_net[i], patch_generator, seg_block) in ``dtype``; ``skip`` is concatenated
    to ``x`` along the channels first (pipeline.py:372).  ``seg_module``: the 1x1 seg_block that will be applied to this
    block's result -- the slab image branch computes it in the block's last epilogue (result attribute ``_cp_seg``)."""
    if _IMG_REUSE is not None and id(module) in _IMG_REUSE:
        return _IMG_REUSE[id(module)]
    if dtype == torch.bfloat16 and _IMAGE_BRANCH == "cudnn":
        y = _bf16_module(module)(x.to(torch.bfloat16), None if skip is None else skip.to(torch.bfloat16))
    elif dtype == torch.bfloat16:
        seq = _tc_module(module)
        y = seq(x, skip, seg=_seg_weights(seg_module)) if seg_module is not None else seq(x, skip)
    else:
        y = _x3_module(module)(x.float(), None if skip is None else skip.float())
    if _IMG_REUSE is not None:
        _IMG_REUSE[id(module)] = y
    return y


def patches_nhwc(patch_generator, img_feat, dtype):
    p = image_block(patch_generator, img_feat, dtype)  # (B,E,Hp,Wp)
    return p.permute(0, 2, 3, 1).contiguous()


# --------------------------------------------------------------------------------------------------
# refine stage (Refine_moduleGNN.forward, pipeline.py:262-298)
# --------------------------------------------------------------------------------------------------
def check_bf16_refine_widths(ref):
    """Raise for a refine stage whose widths the bf16 kernels cannot run, even padded (before any launch)."""
    d0 = ref.pre_graph_module[0].weight.shape[0]
    E = ref.local_feat_ext_block.patch_generator.out_channels
    if d0 % 4 != 0 or 4 * E != d0:
        raise RuntimeError(f"bf16 mode needs query_dims[0] divisible by 4 (the patch embedding is query_dims[0] // 4); got "
                           f"query_dims[0] = {d0}; use float32 mode")
    check_bf16_width("query_dims[0]", d0)
    check_bf16_width("the incoming graph feature", ref.pre_graph_module[0].weight.shape[1] - 4 * E)
    for i in (0, 2, 4):
        check_bf16_width("the query MLP", max(ref.query_block.mlps[i].weight.shape))


def refine_node_major(ref, img_feat, gfeat_nm, roi_mask, x_id, y_id, ctx, dtype, decode=None):
    """One refine stage on plan-order node tensors: gfeat_nm (B,N,Cg) of ``dtype``, roi_mask (B,N) f32 {0,1}, ids (B,N)
    int64, ctx = graph_ctx of the stage's graph (None when it has no graph modules).
    -> logits (B,N,>=2) f32 [x_new, y_new], graph feature (B,N,C) of ``dtype`` (bf16: C = pad64(query_dims[0]), the padded
    channels zero; gfeat_nm may come padded or at its true width).
    ``decode`` = dict(plane, Ltot, x_bits, y_bits, perm, sel[, x_id_kp, y_id_kp]): in bf16 mode the stage's tail (query layers 2
    and 3 + the decode of pipeline.py:375-381, ids updated IN PLACE) runs as one launch (cp_query_decode_fwd) and the returned
    logits are None."""
    _require_eval(ref)
    B, N, Cg = gfeat_nm.shape
    dev = gfeat_nm.device
    k = ref.local_feat_ext_block.kernel_size
    if dtype == torch.bfloat16:
        check_bf16_refine_widths(ref)
    patches = patches_nhwc(ref.local_feat_ext_block.patch_generator, img_feat, dtype)
    slope = float(ref.pre_graph_module[1].negative_slope)
    blocks = list(ref.pre_query_block)
    qmods = [ref.query_block.mlps[i] for i in (0, 2, 4)]
    qslope = float(ref.query_block.mlps[1].negative_slope)
    x_id = x_id.contiguous()
    y_id = y_id.contiguous()
    if dtype == torch.float32:
        pg0 = prepared_linear(ref.pre_graph_module[0], dtype)
        pg1 = prepared_linear(ref.pre_graph_module[2], dtype)
        q = [prepared_linear(m, dtype) for m in qmods]
        taps = ops.sample_taps(patches, x_id, y_id, roi_mask, k)
        h = linear32(taps, pg0, True, slope, a2=gfeat_nm)
        h = linear32(h, pg1, True, slope)
        for blk in blocks:
            h = edgeconv_node_major(blk, h, ctx, dtype)
        t = linear32(h, q[0], True, qslope)
        t = linear32(t, q[1], True, qslope)
        logits = linear32(t, q[2])
        return logits, h
    # ---- bf16 fused kernels, widths padded (see the width notes at the top) ----
    E = patches.shape[-1]
    d0 = ref.pre_graph_module[0].weight.shape[0]
    cg = ref.pre_graph_module[0].weight.shape[1] - 4 * E          # true width of the incoming graph feature
    Ep, cgp = pad16(E), pad64(cg)
    if Ep != E:
        patches = F.pad(patches, (0, Ep - E))
    gfeat_nm = _pad_to(gfeat_nm, cgp)
    pg0 = prepared_linear(ref.pre_graph_module[0], dtype, rows=((d0, pad64(d0)),), cols=((E, Ep),) * 4 + ((cg, cgp),))
    pg1 = _padded_linear(ref.pre_graph_module[2], pad64(d0))
    preps = [prepared_edgeconv(b, dtype) for b in blocks]
    for b in blocks:
        _require_eval(b)
    q0 = _padded_linear(qmods[0], pad64(d0))
    q1 = _padded_linear(qmods[1], q0.nout)
    q = [q0, q1, _padded_linear(qmods[2], q1.nout, last=True)]
    pg_layers = [ops.chain_layer(pg0.packed, pg0.b, pg0.kin, pg0.nout, True, slope),
                 ops.chain_layer(pg1.packed, pg1.b, pg1.kin, pg1.nout, True, slope)]
    q_layers = [ops.chain_layer(q[0].packed, q[0].b, q[0].kin, q[0].nout, True, qslope),
                ops.chain_layer(q[1].packed, q[1].b, q[1].kin, q[1].nout, True, qslope),
                ops.chain_layer(q[2].packed, q[2].b, q[2].kin, q[2].nout, False, 0.0)]
    logits = torch.empty((B, N, 16), dtype=torch.float32, device=dev)
    common = dict(B=B, N=N)
    taps_args = dict(prologue=ops.PRO_TAPS, patches=patches, tap_step=k, x_id=x_id, y_id=y_id, mask=roi_mask,
                     graph_feat=gfeat_nm)
    if not blocks:
        feat = torch.empty((B, N, pg1.nout), dtype=torch.bfloat16, device=dev)
        ops.chain_fwd(**common, **taps_args, layers=pg_layers, out=feat, out_mode=ops.OUT_BF16)
        ops.chain_fwd(**common, prologue=ops.PRO_LOAD, src=feat, layers=q_layers, out=logits, out_mode=ops.OUT_F32,
                      n_valid=q[2].nout)
        return logits, feat
    # K3 + pre-graph MLP + first [P|Q] GEMM in one launch
    z = torch.empty((B, N, 2 * preps[0].Co), dtype=torch.bfloat16, device=dev)
    ops.chain_fwd(**common, **taps_args,
                  layers=pg_layers + [ops.chain_layer(preps[0].packed, preps[0].b, preps[0].C, 2 * preps[0].Co, False, 0.0)],
                  out=z, out_mode=ops.OUT_BF16)
    # EdgeConv j aggregation fused with EdgeConv j+1's [P|Q] GEMM
    for j in range(1, len(blocks)):
        z2 = torch.empty((B, N, 2 * preps[j].Co), dtype=torch.bfloat16, device=dev)
        _agg_gemm(z, ctx, preps[j - 1].slope,
                  ops.chain_layer(preps[j].packed, preps[j].b, preps[j].C, 2 * preps[j].Co, False, 0.0), z2, ops.OUT_BF16)
        z = z2
    # last aggregation (stored: it is the next stage's graph feature) fused with the first query layer, then the rest
    feat = torch.empty((B, N, preps[-1].Co), dtype=torch.bfloat16, device=dev)
    hq = torch.empty((B, N, q[0].nout), dtype=torch.bfloat16, device=dev)
    _agg_gemm(z, ctx, preps[-1].slope, q_layers[0], hq, ops.OUT_BF16, a_out=feat)
    if decode is not None and q[1].nout == 64 and q[2].nout == 2 and q[1].kin in (64, 128, 256):
        ops.query_decode_fwd(src=hq, w1_packed=q[1].packed, b1=q[1].b, slope=qslope, w2=q[2].w, b2=q[2].b, plane=decode["plane"],
                             Ltot=decode["Ltot"], x_bits=decode["x_bits"], y_bits=decode["y_bits"], x_id=x_id, y_id=y_id,
                             perm=decode["perm"], graph_sel=decode["sel"], x_id_kp=decode.get("x_id_kp"), y_id_kp=decode.get("y_id_kp"))
        return None, feat
    ops.chain_fwd(**common, prologue=ops.PRO_LOAD, src=hq, layers=q_layers[1:], out=logits, out_mode=ops.OUT_F32,
                  n_valid=q[2].nout)
    return logits, feat


# --------------------------------------------------------------------------------------------------
# ablation variant without progressive refinement (pipeline_lm.py:286-339, 430-517)
# --------------------------------------------------------------------------------------------------
def mlp_node_major(mods, x_nm, dtype, out_f32=False):
    """nn.Sequential of Linear / LeakyReLU (get_MLP_leakyReLU_layers) on node-major x (B,N,C) of ``dtype``.
    bf16: chain kernel, up to three layers per launch; ``out_f32`` -> (B,N,>=nout padded to 16) f32 logits, else a bf16
    result whose width is padded to a multiple of 64 (zeros beyond nout); x_nm may come padded the same way."""
    mods = list(mods)
    layers = []
    i = 0
    while i < len(mods):
        act = i + 1 < len(mods) and isinstance(mods[i + 1], nn.LeakyReLU)
        layers.append((mods[i], act, float(mods[i + 1].negative_slope) if act else 0.0))
        i += 2 if act else 1
    B, N, _ = x_nm.shape
    if dtype == torch.float32:
        x = x_nm
        for lin, act, slope in layers:
            pl = prepared_linear(lin, dtype)
            x = linear32(x, pl, act, slope)
        return x
    x = _pad_to(x_nm, pad64(layers[0][0].weight.shape[1]))
    for j0 in range(0, len(layers), 3):
        grp = layers[j0:j0 + 3]
        last = j0 + 3 >= len(layers)
        pls, kin = [], x.shape[-1]
        for jj, (lin, _, _) in enumerate(grp):
            pls.append(_padded_linear(lin, kin, last=last and out_f32 and jj == len(grp) - 1))
            kin = pls[-1].nout
        cl = [ops.chain_layer(pl.packed, pl.b, pl.kin, pl.nout, act, slope) for pl, (_, act, slope) in zip(pls, grp)]
        if last and out_f32:
            out = torch.empty((B, N, (pls[-1].nout + 15) // 16 * 16), dtype=torch.float32, device=x.device)
            ops.chain_fwd(prologue=ops.PRO_LOAD, B=B, N=N, src=x, layers=cl, out=out, out_mode=ops.OUT_F32, n_valid=pls[-1].nout)
        else:
            out = torch.empty((B, N, pls[-1].nout), dtype=torch.bfloat16, device=x.device)
            ops.chain_fwd(prologue=ops.PRO_LOAD, B=B, N=N, src=x, layers=cl, out=out, out_mode=ops.OUT_BF16)
        x = out
    return x


def abwoprog_refine_node_major(ref, gfeat_nm, ctx, dtype):
    """Refine_moduleGNN_ABwoProg.forward (pipeline_lm.py:324-339) on plan-order node tensors: MLP on the graph
    feature, then the EdgeConv stack."""
    _require_eval(ref)
    h = mlp_node_major(ref.pre_graph_module, gfeat_nm, dtype)
    for blk in ref.pre_query_block:
        h = edgeconv_node_major(blk, h, ctx, dtype)
    return h


def abwoprog_head_forward(net, img_feats, obj_ids, stage=None, dtype=None):
    """PoseNet_GNNskip_ABwoProg.forward after the backbone (pipeline_lm.py:484-517) -> the reference's 6-tuple."""
    dtype = dtype or get_compute_dtype()
    _require_eval(net)
    nact = net.num_refine_steps if stage is None else stage
    feat_last = img_feats[-1]
    B, dev = feat_last.shape[0], feat_last.device
    _, gfeat, ctx = init_head_node_major(net.init_net, feat_last, obj_ids, dtype)
    img_feat = feat_last
    for i in range(nact):
        img_feat = image_block(net.up_net[i], img_feat, dtype, skip=img_feats[-i - 1] if i > 0 else None)
        sctx = _stage_ctx(net, net.refine_net[i], obj_ids, B, dev, ctx)
        if ctx is None and sctx is not None:      # init net without graph modules: enter the plan order here
            gfeat = sctx.to_plan(gfeat)
        ctx = sctx if sctx is not None else ctx
        gfeat = abwoprog_refine_node_major(net.refine_net[i], gfeat, ctx, dtype)
    seg = image_block(net.seg_block, img_feat, dtype).float().contiguous()
    nb = net.num_bits
    bits = mlp_node_major(net.query_block.mlps, gfeat, dtype, out_f32=True)[:, :, :nb].contiguous()
    if ctx is not None:
        bits = ctx.to_keypoints(bits)
    bits = bits.permute(0, 2, 1).contiguous()      # (B, #bits, N)
    L = net.res_log2
    roi_bit, x_bits, y_bits = bits[:, 0:1], bits[:, 1:L + 1], bits[:, L + 1:]
    x_id = ops.bits_to_id(x_bits, 1, binarize=True, thr=0.0)     # from_code_prob_to_id: sigmoid(x) > 0.5 == x > 0
    y_id = ops.bits_to_id(y_bits, 1, binarize=True, thr=0.0)
    return roi_bit, x_bits, y_bits, seg, x_id, y_id


def _stage_ctx(net, ref, obj_ids, B, dev, base_ctx):
    """GraphCtx of a refine stage; all graphs of one net must share the keypoint renumbering."""
    blocks = list(ref.pre_query_block)
    if not blocks:
        return base_ctx
    ctx = graph_ctx(blocks[0]._knn, obj_ids, B, dev)
    if base_ctx is not None and ctx.plan is not base_ctx.plan:
        # checked once per pair of plans (torch.equal synchronises the stream: a check per step stalled the host three
        # times per step)
        key = (id(ctx.plan), id(base_ctx.plan))
        ok = net.__dict__.setdefault("_cp_perm_ok", {})
        if key not in ok:
            if len(ok) > 64:
                ok.clear()
            ok[key] = (bool(torch.equal(ctx.plan.perm, base_ctx.plan.perm)), ctx.plan, base_ctx.plan)   # keeps the ids alive
        if not ok[key][0]:
            raise RuntimeError("the kNN graphs of one net must be built from the same keypoints (their plan orders differ)")
    return ctx


# --------------------------------------------------------------------------------------------------
# whole progressive head (PoseNet_GNNskip.forward after the backbone, pipeline.py:351-384)
# --------------------------------------------------------------------------------------------------
def pose_head_forward(net, img_feats, obj_ids=None, stage=None, dtype=None, bbox=None, packed=False):
    """-> (roi_bit (B,1,N), x_bits (B,L,N), y_bits (B,L,N), seg (B,2,H,W), x_id (B,N), y_id (B,N)) as the reference,
    plus correspondence records when ``bbox`` (B,4) is given (else None): (B,N,3) int32 {u, v, flags}, or with
    ``packed`` the (B, 16 + 2N) uint8 rows of cp_correspondences_pack (2 bytes per keypoint: what crosses NVLink / PCIe).
    Only ``img_feats[-1], [-2], [-3]`` are read (pipeline.py:361,372): a list of the three deepest maps is enough."""
    dtype = dtype or get_compute_dtype()
    _require_eval(net)
    nact = net.num_refine_steps if stage is None else stage
    feat_last = img_feats[-1]
    B, dev, N = feat_last.shape[0], feat_last.device, net.npoint
    logits0, gfeat, ctx0 = init_head_node_major(net.init_net, feat_last, obj_ids, dtype)
    if ctx0 is None and nact > 0:      # init net without graph modules: take the renumbering of the first refine graph
        ctx0 = _stage_ctx(net, net.refine_net[0], obj_ids, B, dev, None)
        if ctx0 is not None:
            logits0, gfeat = ctx0.to_plan(logits0), ctx0.to_plan(gfeat)
    perm = None if ctx0 is None or ctx0.plan.identity else ctx0.plan.perm
    sel = None if ctx0 is None else ctx0.sel
    L0 = (net.init_net.num_out_bits - 1) // 2
    Ltot = L0 + nact
    roi_bit = torch.empty((B, 1, N), dtype=torch.float32, device=dev)
    x_bits = torch.empty((B, Ltot, N), dtype=torch.float32, device=dev)
    y_bits = torch.empty((B, Ltot, N), dtype=torch.float32, device=dev)
    roi_mask = torch.empty((B, N), dtype=torch.float32, device=dev)   # plan order, like the ids below
    x_id = torch.empty((B, N), dtype=torch.int64, device=dev)
    y_id = torch.empty((B, N), dtype=torch.int64, device=dev)
    ops.decode_init(logits0, L0, Ltot, roi_bit, x_bits, y_bits, roi_mask, x_id, y_id, perm, sel)
    img_feat = feat_last
    for i in range(nact):
        img_feat = image_block(net.up_net[i], img_feat, dtype, skip=img_feats[-i - 1] if i > 0 else None,
                               seg_module=net.seg_block if i == nact - 1 else None)
        ctx = _stage_ctx(net, net.refine_net[i], obj_ids, B, dev, ctx0)
        last_kp = perm is not None and i == nact - 1     # last stage: the ids the caller sees, in keypoint order
        x_kp, y_kp = (torch.empty_like(x_id), torch.empty_like(y_id)) if last_kp else (None, None)
        decode = dict(plane=L0 + i, Ltot=Ltot, x_bits=x_bits, y_bits=y_bits, perm=perm, sel=sel, x_id_kp=x_kp, y_id_kp=y_kp)
        logits, gfeat = refine_node_major(net.refine_net[i], img_feat, gfeat, roi_mask, x_id, y_id, ctx, dtype, decode=decode)
        if logits is not None:      # the stage's tail did not fuse the decode (float32 mode, unusual query dims)
            ops.decode_refine(logits, L0 + i, Ltot, x_bits, y_bits, x_id, y_id, perm, sel, x_kp, y_kp)
        if last_kp:
            x_id, y_id = x_kp, y_kp
    if perm is not None and nact == 0:
        x_id = ops.permute_rows(x_id.view(B, N, 1), perm, sel, True).view(B, N)
        y_id = ops.permute_rows(y_id.view(B, N, 1), perm, sel, True).view(B, N)
    seg = getattr(img_feat, "_cp_seg", None)         # fused into the last up_net convolution's epilogue (slab image branch)
    if seg is None:
        seg = image_block(net.seg_block, img_feat, dtype).float().contiguous()
    corr = None
    if bbox is not None:
        corr = (ops.correspondences_packed if packed else ops.correspondences)(roi_bit, seg, bbox, x_id, y_id)
    return (roi_bit, x_bits, y_bits, seg, x_id, y_id), corr
