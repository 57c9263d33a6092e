"""Tensor-level wrappers over the C ABI (include/checkerpose_b200.h).

PyTorch is used for device memory (``torch.empty``) and the current CUDA stream only; every
computation below is one or more launches of the hand-written kernels in ``csrc/``.  Inputs must be
CUDA tensors: there is no CPU path.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import ChainLayer, ChainParams, ConvBf16Params, ConvSlabParams, EdgeConvParams, GemmX3Params, GraphPlanStruct, QueryDecodeParams, check, lib

CP_F32, CP_BF16 = 0, 1
PRO_LOAD, PRO_AGG, PRO_TAPS = 0, 1, 2
OUT_BF16, OUT_F32 = 0, 1

#: number of kernel launches issued through this module (bench.py reports it as ``gpu_launches``)
launch_count = 0
#: when set to a list, every launch of the tcgen05 GEMM kernels appends (signature, start_event, end_event) (bench.py roofline)
chain_event_log = None


def _count(n=1):
    global launch_count
    launch_count += n


def _timed_launch(fn, name, p, sig):
    """One launch of ``fn(&p, stream)``; with chain_event_log set, CUDA events on the launching stream around it are
    logged under ``sig``."""
    if chain_event_log is None:
        check(fn(C.byref(p), _stream()), name)
    else:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        check(fn(C.byref(p), _stream()), name)
        e1.record()
        chain_event_log.append((sig, e0, e1))
    _count()


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _need_cuda(*tensors):
    """Every tensor of a launch must be a CUDA tensor on ONE device, and that device must be the current one: the
    kernels are launched on ``torch.cuda.current_stream()``, i.e. on the current device (wrap calls for another GPU in
    ``with torch.cuda.device(t.device):`` -- the module-level forwards do)."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("checkerpose_b200: expected a CUDA tensor (there is no CPU fallback); got device "
                               f"{t.device}")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"checkerpose_b200: tensors of one launch live on different devices ({dev} and {t.device})")
    if dev is not None and dev.index != torch.cuda.current_device():
        raise RuntimeError(f"checkerpose_b200: tensors live on {dev} but the current CUDA device is cuda:{torch.cuda.current_device()}; "
                           "wrap the call in `with torch.cuda.device(...)`")


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return CP_F32
    if t.dtype == torch.bfloat16:
        return CP_BF16
    raise RuntimeError(f"checkerpose_b200: unsupported dtype {t.dtype}")


def _p(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


# ------------------------------------------------------------------------------------------------ K1
def knn(x: torch.Tensor, k: int, want_i32: bool = False):
    """x (B,C,N) float32 -> idx (B,N,k) int64 [, int32 copy].  pipeline.py:18-23."""
    _need_cuda(x)
    if x.dim() != 3:
        raise RuntimeError("knn: x must be (B, C, N)")
    x = x.contiguous().float()
    B, Cc, N = x.shape
    idx = torch.empty((B, N, k), dtype=torch.int64, device=x.device)
    idx32 = torch.empty((B, N, k), dtype=torch.int32, device=x.device) if want_i32 else None
    check(lib.cp_knn(_p(x), B, Cc, N, int(k), _p(idx), _p(idx32), _stream()), "cp_knn")
    _count()
    return (idx, idx32) if want_i32 else idx


# --------------------------------------------------------------------------------------- layout
def is_node_major_view(x: torch.Tensor) -> bool:
    """True if the (B,C,N) tensor is a permuted view of contiguous (B,N,C) storage."""
    return x.dim() == 3 and x.permute(0, 2, 1).is_contiguous()


def to_node_major(x: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """(B,C,N) -> contiguous (B,N,C) of ``dtype``; zero-copy when x already is such a view."""
    _need_cuda(x)
    B, Cc, N = x.shape
    if is_node_major_view(x):
        v = x.permute(0, 2, 1)
        if v.dtype == dtype:
            return v
        out = torch.empty((B, N, Cc), dtype=dtype, device=x.device)
        check(lib.cp_convert(_p(v), _dt(v), _p(out), _dt(out), v.numel(), _stream()), "cp_convert")
        _count()
        return out
    x = x.contiguous()
    out = torch.empty((B, N, Cc), dtype=dtype, device=x.device)
    check(lib.cp_transpose_cn_to_nc(_p(x), _dt(x), _p(out), _dt(out), B, Cc, N, _stream()), "cp_transpose_cn_to_nc")
    _count()
    return out


def to_channel_major(x: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """contiguous (B,N,C) -> contiguous (B,C,N) of ``dtype``."""
    _need_cuda(x)
    x = x.contiguous()
    B, N, Cc = x.shape
    out = torch.empty((B, Cc, N), dtype=dtype, device=x.device)
    check(lib.cp_transpose_nc_to_cn(_p(x), _dt(x), _p(out), _dt(out), B, N, Cc, _stream()), "cp_transpose_nc_to_cn")
    _count()
    return out


def transpose_scatter(x: torch.Tensor, bias=None, row_map=None, graph_sel=None) -> torch.Tensor:
    """contiguous bf16 (B,R,S) -> (B,S,R) with out[b, row_map[g(b)][s], r] = x[b, r, s] + bias[s] (cp_transpose_scatter_bf16)."""
    _need_cuda(x, bias, row_map, graph_sel)
    assert x.dtype == torch.bfloat16 and x.is_contiguous()
    B, R, S = x.shape
    out = torch.empty((B, S, R), dtype=torch.bfloat16, device=x.device)
    check(lib.cp_transpose_scatter_bf16(_p(x), _p(out), B, R, S, _p(bias), _p(row_map), _p(graph_sel), _stream()),
          "cp_transpose_scatter_bf16")
    _count()
    return out


def bias_add_rows_(x: torch.Tensor, bias: torch.Tensor, relu: bool = False) -> torch.Tensor:
    """x (..., C) bf16, channels contiguous: x = [relu](x + bias (C) f32) in place (cp_bias_add_rows_bf16)."""
    _need_cuda(x, bias)
    assert x.dtype == torch.bfloat16 and x.is_contiguous() and bias.dtype == torch.float32 and bias.is_contiguous()
    Cc = x.shape[-1]
    check(lib.cp_bias_add_rows_bf16(_p(x), _p(bias), x.numel() // Cc, Cc, int(bool(relu)), _stream()), "cp_bias_add_rows_bf16")
    _count()
    return x


def convert(x: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    _need_cuda(x)
    if x.dtype == dtype:
        return x
    x = x.contiguous()
    out = torch.empty(x.shape, dtype=dtype, device=x.device)
    check(lib.cp_convert(_p(x), _dt(x), _p(out), _dt(out), x.numel(), _stream()), "cp_convert")
    _count()
    return out


def graph_feature(x: torch.Tensor, idx32: torch.Tensor, graph_sel=None) -> torch.Tensor:
    """get_graph_feature (pipeline.py:27-40): x (B,C,N) f32 -> (B,2C,N,K) f32."""
    _need_cuda(x, idx32, graph_sel)
    x = x.contiguous().float()
    B, Cc, N = x.shape
    K = idx32.shape[-1]
    out = torch.empty((B, 2 * Cc, N, K), dtype=torch.float32, device=x.device)
    check(lib.cp_graph_feature(_p(x), _p(idx32), _p(graph_sel), _p(out), B, Cc, N, K, _stream()), "cp_graph_feature")
    _count()
    return out


# ------------------------------------------------------------------------------- weight preparation
def fold_edgeconv(conv_w, gamma, beta, mean, var, eps=1e-5):
    """-> (w_fold (2Co,C) f32, b_fold (2Co) f32); see cp_fold_edgeconv in the header for the algebra."""
    _need_cuda(conv_w, gamma, beta, mean, var)
    Co, C2 = conv_w.shape[0], conv_w.shape[1]
    Cc = C2 // 2
    w = conv_w.reshape(Co, C2).contiguous().float()
    wf = torch.empty((2 * Co, Cc), dtype=torch.float32, device=w.device)
    bf = torch.empty((2 * Co,), dtype=torch.float32, device=w.device)
    check(lib.cp_fold_edgeconv(_p(w), _p(gamma.contiguous().float()), _p(beta.contiguous().float()),
                               _p(mean.contiguous().float()), _p(var.contiguous().float()), float(eps), Cc, Co,
                               _p(wf), _p(bf), _stream()), "cp_fold_edgeconv")
    _count()
    return wf, bf


def pack_weight(w: torch.Tensor) -> torch.Tensor:
    """(Nout,K) f32 -> packed bf16 tile image (uint8 tensor) for the tcgen05 chain kernel."""
    _need_cuda(w)
    w = w.contiguous().float()
    Nout, K = w.shape
    nbytes = lib.cp_packed_weight_bytes(Nout, K)
    if nbytes == 0:
        raise RuntimeError(f"pack_weight: unsupported shape ({Nout},{K}); K must be a multiple of 64")
    out = torch.empty((nbytes,), dtype=torch.uint8, device=w.device)
    check(lib.cp_pack_weight(_p(w), Nout, K, _p(out), _stream()), "cp_pack_weight")
    _count()
    return out


# ------------------------------------------------------------------- float32 mode on tcgen05 (split bf16 x 3)
X3_LINEAR, X3_CONV, X3_CONVT = 0, 1, 2


def pack_weight_split(w: torch.Tensor):
    """(Nout,K) f32 -> (packed bf16(w), packed bf16(w - bf16(w))) tile images for cp_gemm_x3."""
    _need_cuda(w)
    w = w.contiguous().float()
    Nout, K = w.shape
    nbytes = lib.cp_packed_weight_bytes(Nout, K)
    if nbytes == 0:
        raise RuntimeError(f"pack_weight_split: unsupported shape ({Nout},{K}); K must be a multiple of 64")
    hi = torch.empty((nbytes,), dtype=torch.uint8, device=w.device)
    lo = torch.empty((nbytes,), dtype=torch.uint8, device=w.device)
    check(lib.cp_pack_weight_split(_p(w), Nout, K, _p(hi), _p(lo), _stream()), "cp_pack_weight_split")
    _count()
    return hi, lo


def gemm_x3_linear(a1, w_split, nout, bias=None, act=False, slope=0.0, a2=None, out=None):
    """y = act([a1|a2] @ W.T + bias) in float32 on the tensor cores (cp_gemm_x3, CP_X3_LINEAR); a* (..., K*) fp32 rows."""
    _need_cuda(a1, a2, bias, w_split[0], w_split[1])
    assert a1.dtype == torch.float32 and a1.stride(-1) == 1
    a1 = a1 if a1.is_contiguous() else a1.contiguous()
    K1 = a1.shape[-1]
    M = a1.numel() // K1
    K2 = 0
    if a2 is not None:
        assert a2.dtype == torch.float32
        a2 = a2 if a2.is_contiguous() else a2.contiguous()
        K2 = a2.shape[-1]
    if out is None:
        out = torch.empty(a1.shape[:-1] + (nout,), dtype=torch.float32, device=a1.device)
    p = GemmX3Params()
    p.mode = X3_LINEAR
    p.a1, p.ld1, p.k1 = _p(a1), K1, K1
    p.a2, p.ld2, p.k2 = _p(a2), K2, K2
    p.M, p.K = M, K1 + K2
    p.w_hi, p.w_lo = _p(w_split[0]), _p(w_split[1])
    p.bias, p.act, p.slope = _p(bias), int(bool(act)), float(slope)
    p.out, p.ld_out, p.Nout = _p(out), out.stride(-2) if out.dim() > 1 else nout, int(nout)
    _timed_launch(lib.cp_gemm_x3, "cp_gemm_x3", p, ("X3", K1 + K2, (int(nout),), OUT_F32, M, 0))
    return out


def _conv_gemm_params(p, x_nhwc, dtype, nout, KH, KW, pad, Ho, Wo, bias, act, slope, transposed):
    """Fill the fields cp_gemm_x3_params and cp_conv_bf16_params share for Conv2d KH x KW stride 1 / ConvTranspose2d stride 2
    of the NHWC map x_nhwc (B,H,W,Cin) of ``dtype`` -> the (B,Ho,Wo,nout) output map of ``dtype``."""
    assert x_nhwc.dtype == dtype and x_nhwc.is_contiguous() and x_nhwc.dim() == 4
    B, H, W, Cin = x_nhwc.shape
    out = torch.empty((B, Ho, Wo, nout), dtype=dtype, device=x_nhwc.device)
    p.mode = X3_CONVT if transposed else X3_CONV
    p.a1, p.ld1, p.k1 = _p(x_nhwc), Cin, Cin
    p.H, p.W, p.Ho, p.Wo, p.KH, p.KW, p.pad = H, W, int(Ho), int(Wo), int(KH), int(KW), int(pad)
    p.M, p.K = B * Ho * Wo, KH * KW * Cin
    p.bias, p.act, p.slope = _p(bias), int(bool(act)), float(slope)
    p.out, p.ld_out, p.Nout = _p(out), int(nout), int(nout)
    return out


def gemm_x3_conv(x_nhwc, w_split, nout, KH, KW, pad, Ho, Wo, bias=None, act=False, slope=0.0, transposed=False):
    """Conv2d KH x KW stride 1 / ConvTranspose2d stride 2 over an fp32 NHWC map (B,H,W,Cin) -> (B,Ho,Wo,nout) fp32, as an
    implicit GEMM on the tensor cores (cp_gemm_x3, CP_X3_CONV / CP_X3_CONVT); W rows in (ky, kx, c) order."""
    _need_cuda(x_nhwc, bias, w_split[0], w_split[1])
    p = GemmX3Params()
    out = _conv_gemm_params(p, x_nhwc, torch.float32, nout, KH, KW, pad, Ho, Wo, bias, act, slope, transposed)
    p.w_hi, p.w_lo = _p(w_split[0]), _p(w_split[1])
    _timed_launch(lib.cp_gemm_x3, "cp_gemm_x3", p, ("X3C", p.K, (int(nout),), OUT_F32, p.M, 0))
    return out


# ------------------------------------------------------------------- bf16 implicit-GEMM convolution on tcgen05
def conv_bf16(x_nhwc, w_packed, nout, KH, KW, pad, Ho, Wo, bias=None, act=False, slope=0.0, transposed=False):
    """Conv2d KH x KW stride 1 / ConvTranspose2d stride 2 over a bf16 NHWC map (B,H,W,Cin) -> (B,Ho,Wo,nout) bf16 as an implicit
    GEMM on the tensor cores (cp_conv_bf16); W rows in (ky, kx, c) order, packed by pack_weight."""
    _need_cuda(x_nhwc, bias, w_packed)
    p = ConvBf16Params()
    out = _conv_gemm_params(p, x_nhwc, torch.bfloat16, nout, KH, KW, pad, Ho, Wo, bias, act, slope, transposed)
    p.w_packed = _p(w_packed)
    _timed_launch(lib.cp_conv_bf16, "cp_conv_bf16", p, ("CV", p.K, (int(nout),), OUT_BF16, p.M, 0))
    return out


# ------------------------------------------------------------------- slab convolutions over zero-bordered maps
def _slab_common(xp, w_packed, K, nout, bias, act, slope):
    _need_cuda(xp, bias, w_packed)
    assert xp.dtype == torch.bfloat16 and xp.is_contiguous() and xp.dim() == 4
    B, Hp, Wp, Cin = xp.shape
    p = ConvSlabParams()
    p.x, p.B, p.Hp, p.Wp, p.C, p.ldx = _p(xp), B, Hp, Wp, Cin, Cin
    p.w_packed, p.K = _p(w_packed), int(K)
    p.bias, p.act, p.slope = _p(bias), int(bool(act)), float(slope)
    p.Nout = int(nout)
    return p


def _slab_grid_taps(p, KH, KW, Wp, cy, cx):
    """One phase of KH x KW taps over the stored grid: tap (ky, kx) reads the row shift (ky - cy) * Wp + (kx - cx)."""
    p.num_phases = 1
    ph = p.phase[0]
    ph.ntaps = KH * KW
    for ky in range(KH):
        for kx in range(KW):
            t = ky * KW + kx
            ph.wtap[t] = t
            ph.shift[t] = (ky - cy) * Wp + (kx - cx)
    p.compact = 0


def zero_border(xp):
    """Zero the shared border (last row and last column of every image) of a stored NHWC map (B,H+1,W+1,C) in place."""
    _need_cuda(xp)
    assert xp.is_contiguous() and xp.dim() == 4
    B, Hp, Wp, Cc = xp.shape
    check(lib.cp_zero_border_nhwc(_p(xp), B, Hp, Wp, Cc, xp.element_size(), _stream()), "cp_zero_border_nhwc")
    _count()
    return xp


# Bordered layout of the slab convolutions: an image (H, W) is stored as (H+1, W+1) with a zero LAST row and LAST column.
# Over the flat pixel index of the whole batch that one column is the right border of its row and the left border of the
# next one, the one row is the bottom border of its image and the top border of the next one; the rows before the first
# image and after the last one are zero-filled by the TMA unit.  (H+1)(W+1) / HW = 3 % more rows at 64 x 64.
def to_bordered(x_nhwc):
    """(B,H,W,C) -> the bordered (B,H+1,W+1,C) copy."""
    return torch.nn.functional.pad(x_nhwc, (0, 0, 0, 1, 0, 1))


def _slab_seg(p, seg, B, Hp, Wp, nout, dev):
    """Attach the fused 1x1 head (seg = (weight (n, nout) f32, bias (n,) f32)) -> its (B, n, H, W) f32 output."""
    if seg is None:
        return None
    sw, sb = seg
    _need_cuda(sw, sb)
    assert sw.dtype == torch.float32 and sb.dtype == torch.float32 and sw.is_contiguous() and sw.shape == (sb.shape[0], nout) and sw.shape[0] <= 4
    seg_out = torch.empty((B, sw.shape[0], Hp - 1, Wp - 1), dtype=torch.float32, device=dev)
    p.seg_w, p.seg_b, p.seg_out, p.seg_n = _p(sw), _p(sb), _p(seg_out), int(sw.shape[0])
    return seg_out


def conv_slab_same(xp, w_packed, nout, KH, KW, bias=None, act=False, slope=0.0, seg=None):
    """Conv2d KH x KW (1 or 3), stride 1, "same" padding, over a bordered bf16 map xp (B, H+1, W+1, Cin) -> the bordered
    (B, H+1, W+1, nout) map of the result (its border written as zeros): chains of such convolutions never leave the
    layout.  W rows in (ky, kx, c) order, packed by pack_weight.  seg = (weight (n, nout), bias (n,)) f32 fuses a 1x1
    convolution of the result (seg_block) into the epilogue: returns (map, (B, n, H, W) f32)."""
    B, Hp, Wp, Cin = xp.shape
    assert KH % 2 == 1 and KW % 2 == 1 and KH <= 3 and KW <= 3
    p = _slab_common(xp, w_packed, KH * KW * Cin, nout, bias, act, slope)
    seg_out = _slab_seg(p, seg, B, Hp, Wp, nout, xp.device)
    out = torch.empty((B, Hp, Wp, nout), dtype=torch.bfloat16, device=xp.device)
    p.out, p.ld_out = _p(out), int(nout)
    _slab_grid_taps(p, KH, KW, Wp, KH // 2, KW // 2)
    p.vy0, p.vy1, p.vx0, p.vx1 = 0, Hp - 1, 0, Wp - 1
    # signature: ..., rows of the launch, multiply-accumulates of the convolution proper (without the border rows)
    _timed_launch(lib.cp_conv_slab, "cp_conv_slab", p, ("CS", KH * KW * Cin, (int(nout),), OUT_BF16, B * Hp * Wp, B * (Hp - 1) * (Wp - 1) * KH * KW * Cin * int(nout)))
    return out if seg is None else (out, seg_out)


def conv_slab_full(xp, w_packed, nout, KH, KW, bias=None, act=False, slope=0.0):
    """Conv2d 2 x 2, stride 1, padding 1 (patch_generator, pipeline.py:144-145) over a bordered bf16 map xp (B, H+1, W+1, Cin)
    -> contiguous (B, H+1, W+1, nout): output (oy, ox) reads pixels (oy-1+ky, ox-1+kx), so the output grid IS the stored grid
    -- every row of the launch is a real output."""
    B, Hp, Wp, Cin = xp.shape
    assert KH == 2 and KW == 2
    p = _slab_common(xp, w_packed, KH * KW * Cin, nout, bias, act, slope)
    out = torch.empty((B, Hp, Wp, nout), dtype=torch.bfloat16, device=xp.device)
    p.out, p.ld_out = _p(out), int(nout)
    _slab_grid_taps(p, KH, KW, Wp, 1, 1)
    p.vy0, p.vy1, p.vx0, p.vx1 = 0, Hp, 0, Wp
    _timed_launch(lib.cp_conv_slab, "cp_conv_slab", p, ("CS", KH * KW * Cin, (int(nout),), OUT_BF16, B * Hp * Wp, B * Hp * Wp * KH * KW * Cin * int(nout)))
    return out


def convT_slab(x_nhwc, w_packed, nout, bias=None, act=False, slope=0.0):
    """ConvTranspose2d(kernel 3, stride 2, padding 1, output_padding 1) (pipeline.py:187-197) of a bf16 NHWC map (B,H,W,Cin)
    as the FOUR output parities of the result, each a small convolution over the input with its own 1 / 2 / 2 / 4 taps (9 tap
    GEMMs in all; the gather formulation of cp_conv_bf16 multiplies 36, three quarters of them zeros).  Returns the
    bordered (B, 2H+1, 2W+1, nout) map.  W rows in (ky, kx, c) order, packed by pack_weight."""
    B, H, W, Cin = x_nhwc.shape
    xp = to_bordered(x_nhwc)
    Hp, Wp = H + 1, W + 1
    p = _slab_common(xp, w_packed, 9 * Cin, nout, bias, act, slope)
    OHp, OWp = 2 * H + 1, 2 * W + 1
    out = torch.empty((B, OHp, OWp, nout), dtype=torch.bfloat16, device=xp.device)
    zero_border(out)
    p.out, p.ld_out = _p(out), int(nout)
    p.num_phases = 4
    # oy = 2 iy - 1 + ky: even rows oy = 2i take ky = 1 from iy = i; odd rows oy = 2i + 1 take ky = 2 from iy = i and ky = 0 from i + 1
    taps1 = {0: [(1, 0)], 1: [(2, 0), (0, 1)]}          # parity -> [(k, input offset)]
    for dy in range(2):
        for dx in range(2):
            ph = p.phase[dy * 2 + dx]
            t = 0
            for ky, sy in taps1[dy]:
                for kx, sx in taps1[dx]:
                    ph.wtap[t] = ky * 3 + kx
                    ph.shift[t] = sy * Wp + sx
                    t += 1
            ph.ntaps = t
            ph.out_off = dy * OWp + dx
    p.vy0, p.vy1, p.vx0, p.vx1 = 0, H, 0, W
    p.compact, p.out_sb, p.out_sy, p.out_sx = 1, OHp * OWp, 2 * OWp, 2
    _timed_launch(lib.cp_conv_slab, "cp_conv_slab", p, ("CS", 9 * Cin, (int(nout),), OUT_BF16, B * Hp * Wp, B * H * W * 9 * Cin * int(nout)))
    return out


def upsample2x_cat_padded(a, b=None):
    """upsample2x_cat writing the interior of a bordered NHWC map: returns (B, 2H+1, 2W+1, Ca+Cb) contiguous."""
    B, Ct, H, W, src = _upsample_sources(a, b)
    out = torch.empty((B, 2 * H + 1, 2 * W + 1, Ct), dtype=a.dtype, device=a.device)
    zero_border(out)
    check(lib.cp_upsample2x_cat_nhwc_to(*src, _p(out), out.stride(0), out.stride(1), out.stride(2), B, H, W, _stream()),
          "cp_upsample2x_cat_nhwc_to")
    _count()
    return out


# ------------------------------------------------------------------------------------ fp32 SIMT path
def linear_f32(a1, w, bias=None, act=False, slope=0.0, a2=None, out=None):
    """y = act([a1|a2] @ w.T + bias); a* are (..., K*) row-major views with unit inner stride."""
    _need_cuda(a1, w, bias, a2)
    K1 = a1.shape[-1]
    M = a1.numel() // K1
    K2 = 0 if a2 is None else a2.shape[-1]
    Nout = w.shape[0]
    assert w.shape[1] == K1 + K2 and a1.stride(-1) == 1
    a1 = a1 if a1.is_contiguous() else a1.contiguous()
    if a2 is not None:
        a2 = a2 if a2.is_contiguous() else a2.contiguous()
    if out is None:
        out = torch.empty(a1.shape[:-1] + (Nout,), dtype=torch.float32, device=a1.device)
    check(lib.cp_linear_f32(_p(a1), K1, K1, _p(a2), K2, K2, _p(w), _p(bias), int(bool(act)), float(slope), _p(out),
                            out.stride(-2) if out.dim() > 1 else Nout, M, Nout, _stream()), "cp_linear_f32")
    _count()
    return out


def edge_aggregate(z, idx32, graph_sel, slope, out=None):
    """z (B,N,2Co) -> y (B,N,Co):  lrelu(max_k z[b,idx[i,k],:Co] + z[b,i,Co:])."""
    _need_cuda(z, idx32, graph_sel)
    B, N, C2 = z.shape
    Co = C2 // 2
    K = idx32.shape[-1]
    assert z.is_contiguous() and idx32.is_contiguous() and idx32.shape[-2] == N
    if out is None:
        out = torch.empty((B, N, Co), dtype=z.dtype, device=z.device)
    check(lib.cp_edge_aggregate(_p(z), _dt(z), _p(idx32), _p(graph_sel), float(slope), _p(out), B, N, K, Co, _stream()),
          "cp_edge_aggregate")
    _count()
    return out


def edge_aggregate_staged(z, plan, graph_sel, slope, out=None):
    """float32 aggregation on the graph plan (cp_edge_aggregate_staged_f32): z (B,N,2Co) fp32 in PLAN order -> (B,N,Co)."""
    _need_cuda(z, graph_sel)
    B, N, C2 = z.shape
    Co = C2 // 2
    assert z.dtype == torch.float32 and z.is_contiguous() and N == plan.N
    if out is None:
        out = torch.empty((B, N, Co), dtype=torch.float32, device=z.device)
    check(lib.cp_edge_aggregate_staged_f32(_p(z), C.byref(plan.struct), _p(graph_sel), float(slope), _p(out), B, N, Co, _stream()),
          "cp_edge_aggregate_staged_f32")
    _count()
    return out


def sample_taps(patches_nhwc, x_id, y_id, mask, tap_step, out=None):
    """patches (B,Hp,Wp,E) contiguous, ids (B,N) int64, mask (B,N) f32|None -> (B,N,4E)."""
    _need_cuda(patches_nhwc, x_id, y_id, mask)
    B, Hp, Wp, E = patches_nhwc.shape
    N = x_id.shape[1]
    assert patches_nhwc.is_contiguous() and x_id.is_contiguous() and y_id.is_contiguous()
    assert x_id.dtype == torch.int64 and y_id.dtype == torch.int64
    if out is None:
        out = torch.empty((B, N, 4 * E), dtype=patches_nhwc.dtype, device=patches_nhwc.device)
    check(lib.cp_sample_taps(_p(patches_nhwc), _dt(patches_nhwc), Hp, Wp, E, int(tap_step), _p(x_id), _p(y_id), _p(mask),
                             _p(out), B, N, _stream()), "cp_sample_taps")
    _count()
    return out


def _nhwc_strides(t):
    """(B,C,H,W) tensor whose channel stride is 1 -> element strides (sb, sh, sw)."""
    if t.dim() != 4 or t.stride(1) != 1:
        raise RuntimeError("expected a channels_last (B,C,H,W) tensor")
    return t.stride(0), t.stride(2), t.stride(3)


def _upsample_sources(a, b):
    """Check the sources of the x2 upsampling -> (B, Ca+Cb, H, W, the source arguments of cp_upsample2x_cat_nhwc[_to])."""
    _need_cuda(a, b)
    B, Ca, H, W = a.shape
    Cb = 0 if b is None else b.shape[1]
    if b is not None and (b.shape[0] != B or b.shape[2:] != a.shape[2:] or b.dtype != a.dtype):
        raise RuntimeError("upsample2x_cat: sources disagree in shape or dtype")
    sa = _nhwc_strides(a)
    sb = (0, 0, 0) if b is None else _nhwc_strides(b)
    return B, Ca + Cb, H, W, (_p(a), *sa, Ca, _p(b), *sb, Cb, _dt(a))


def upsample2x_cat(a, b=None):
    """Bilinear x2 (align_corners=True) of cat([a, b], 1) for channels_last (B,C,H,W) inputs.
    Returns a channels_last (B, Ca+Cb, 2H, 2W) tensor (a permuted view of NHWC storage)."""
    B, Ct, H, W, src = _upsample_sources(a, b)
    out = torch.empty((B, 2 * H, 2 * W, Ct), dtype=a.dtype, device=a.device)
    check(lib.cp_upsample2x_cat_nhwc(*src, _p(out), B, H, W, _stream()), "cp_upsample2x_cat_nhwc")
    _count()
    return out.permute(0, 3, 1, 2)


# ------------------------------------------------------------------------------- tcgen05 chain
class _Layer(ChainLayer):
    """ChainLayer that keeps its tensors alive until the launch has been issued."""


def chain_layer(w_packed, bias, kin, nout, act, slope, w_stride=0, b_stride=0) -> ChainLayer:
    """``w_stride`` (bytes) / ``b_stride`` (floats): distance between consecutive objects' packed weights / biases; RoI b of
    a launch then uses object graph_sel[b] (see cp_chain_layer)."""
    L = _Layer(C.c_void_p(w_packed.data_ptr()), _p(bias), int(kin), int(nout), int(bool(act)), float(slope), int(w_stride),
               int(b_stride))
    L._keepalive = (w_packed, bias)
    return L


def chain_fwd(*, prologue, B, N, layers, out, out_mode, n_valid=0,
              src=None, z=None, idx32=None, graph_sel=None, agg_slope=0.2, a_out=None,
              patches=None, tap_step=2, x_id=None, y_id=None, mask=None, graph_feat=None):
    """One launch of the fused tcgen05 chain (see cp_chain_fwd in the header).  All tensors bf16
    node-major unless noted; ``out`` is (B,N,ld) bf16 (OUT_BF16) or f32 (OUT_F32)."""
    _need_cuda(out, src, z, idx32, graph_sel, a_out, patches, x_id, y_id, mask, graph_feat)
    p = ChainParams()
    p.prologue, p.B, p.N = prologue, B, N
    p.graph_sel = _p(graph_sel)      # AGG: the RoI's graph; every prologue: its weights when a layer has strides
    if prologue == PRO_LOAD:
        assert src.dtype == torch.bfloat16 and src.stride(-1) == 1
        p.src, p.ld_src, p.C = _p(src), src.stride(-2), src.shape[-1]
    elif prologue == PRO_AGG:
        assert z.dtype == torch.bfloat16 and z.is_contiguous() and idx32.dtype == torch.int32 and idx32.is_contiguous()
        p.z, p.ld_z, p.Co = _p(z), z.shape[-1], z.shape[-1] // 2
        p.idx, p.K, p.agg_slope = _p(idx32), idx32.shape[-1], float(agg_slope)
        if a_out is not None:
            assert a_out.dtype == torch.bfloat16 and a_out.is_contiguous()
            p.a_out, p.ld_a_out = _p(a_out), a_out.shape[-1]
    elif prologue == PRO_TAPS:
        assert patches.dtype == torch.bfloat16 and patches.is_contiguous() and graph_feat.dtype == torch.bfloat16
        assert x_id.dtype == torch.int64 and y_id.dtype == torch.int64 and graph_feat.is_contiguous()
        p.patches, p.Hp, p.Wp, p.E, p.tap_step = _p(patches), patches.shape[1], patches.shape[2], patches.shape[3], int(tap_step)
        p.x_id, p.y_id, p.mask = _p(x_id), _p(y_id), _p(mask)
        p.graph_feat, p.ld_gf, p.Cg = _p(graph_feat), graph_feat.shape[-1], graph_feat.shape[-1]
    else:
        raise RuntimeError("chain_fwd: bad prologue")
    p.num_layers = len(layers)
    for i, L in enumerate(layers):
        p.layers[i] = L
    p.out_mode, p.out, p.ld_out, p.n_valid = out_mode, _p(out), out.shape[-1], int(n_valid)
    _timed_launch(lib.cp_chain_fwd, "cp_chain_fwd", p, (prologue, layers[0].kin, tuple(L.nout for L in layers), out_mode, B, N))
    return out


# --------------------------------------------------------------------- staged EdgeConv (graph plan)
PLAN_UMAX = 512     # CP_PLAN_UMAX
PLAN_TILE = 128     # CP_PLAN_TILE
PLAN_PAIRS = 64     # CP_PLAN_PAIRS
PLAN_LIST_LANES = 64  # CP_PLAN_LIST_LANES
PLAN_MAX_K = 40


class GraphPlan:
    """Device-resident result of cp_graph_plan_build for a (G,N,K) kNN table (see the header).  ``perm`` maps plan
    position -> keypoint id; ``idx_p`` is the neighbour table in plan numbering; ``ucount`` / ``ulist`` are the distinct
    neighbour rows of every 128-node tile, ``prog`` the tile's 64 node-pair programs; ``staged`` tells whether every
    tile's distinct rows fit the staged kernel's shared-memory ring."""

    def __init__(self, idx32: torch.Tensor, xyz):
        """idx32 (G,N,K) int32 tensor in keypoint numbering (the plan lives on its device); xyz (G,3,N) or None."""
        G, N, K = idx32.shape
        dev = idx32.device
        T = (N + PLAN_TILE - 1) // PLAN_TILE
        KP = int(lib.cp_graph_plan_kp(K))
        idx_h = idx32.cpu().contiguous()
        xyz_h = None if xyz is None else xyz.detach().to("cpu", torch.float32).contiguous()
        if xyz_h is not None and tuple(xyz_h.shape) != (G, 3, N):
            raise RuntimeError(f"GraphPlan: keypoints {tuple(xyz_h.shape)} do not match the graph table {(G, N, K)}")
        self.G, self.N, self.K, self.KP, self.T = G, N, K, KP, T
        if KP < 0:      # K > 40: no plan-order staging; keep the caller's numbering and the unstaged kernel
            self.PW = 0
            self.max_unique = N
            self.staged, self.identity = False, True
            self.perm = torch.arange(N, dtype=torch.int32, device=dev).expand(G, N).contiguous()
            self.perm_inv = self.perm
            self.idx_p = idx32.contiguous()
            self.ucount = self.ulist = self.prog = self.struct = None
            return
        PW = 2 * KP + 8
        perm = torch.empty((G, N), dtype=torch.int32)
        idx_p = torch.empty((G, N, K), dtype=torch.int32)
        ucount = torch.empty((G, T), dtype=torch.int32)
        ulist = torch.empty((G, T, PLAN_LIST_LANES, PLAN_UMAX // PLAN_LIST_LANES), dtype=torch.int16)
        prog = torch.empty((G, T, PLAN_PAIRS, PW), dtype=torch.int16)
        worst = lib.cp_graph_plan_build(_p(xyz_h), _p(idx_h), G, N, K, PLAN_UMAX, _p(perm), _p(idx_p), _p(ucount), _p(ulist),
                                        _p(prog))
        check(min(worst, 0), "cp_graph_plan_build")
        self.PW = PW
        self.max_unique = int(worst)
        self.ring_rows = int(lib.cp_edgeconv_ring_rows(KP))
        self.staged = worst <= min(PLAN_UMAX, self.ring_rows)
        self.identity = bool((perm == torch.arange(N, dtype=torch.int32)).all())
        self.perm = perm.to(dev)
        inv = torch.empty_like(perm)
        inv.scatter_(1, perm.long(), torch.arange(N, dtype=torch.int32).expand(G, N).contiguous())
        self.perm_inv = inv.to(dev)        # keypoint id -> plan position
        self.idx_p = idx_p.to(dev)
        self.ucount, self.ulist, self.prog = ucount.to(dev), ulist.to(dev), prog.to(dev)
        self.struct = GraphPlanStruct(G, N, K, KP, T, PLAN_UMAX, self.max_unique, self.ucount.data_ptr(), self.ulist.data_ptr(),
                                      self.prog.data_ptr())


def edgeconv_fwd(*, z, plan: GraphPlan, graph_sel, agg_slope, layer, out, out_mode, n_valid=0, a_out=None):
    """One launch of the staged EdgeConv kernel (cp_edgeconv_fwd).  z (B,N,2Co) bf16 in plan order."""
    _need_cuda(z, out, a_out, graph_sel)
    if not plan.staged:
        raise RuntimeError("edgeconv_fwd: this graph does not fit the staged kernel (see GraphPlan.staged)")
    assert z.dtype == torch.bfloat16 and z.is_contiguous() and z.shape[1] == plan.N
    p = EdgeConvParams()
    p.B, p.N = z.shape[0], z.shape[1]
    p.z, p.ld_z, p.Co = _p(z), z.shape[-1], z.shape[-1] // 2
    p.plan, p.graph_sel, p.agg_slope = plan.struct, _p(graph_sel), float(agg_slope)
    if a_out is not None:
        assert a_out.dtype == torch.bfloat16 and a_out.is_contiguous()
        p.a_out, p.ld_a_out = _p(a_out), a_out.shape[-1]
    p.layer = layer
    p.out_mode, p.out, p.ld_out, p.n_valid = out_mode, _p(out), out.shape[-1], int(n_valid)
    _timed_launch(lib.cp_edgeconv_fwd, "cp_edgeconv_fwd", p, ("EC", p.Co, (layer.nout,), out_mode, p.B, p.N))
    return out


def graph_sel(obj_ids: torch.Tensor, G: int) -> torch.Tensor:
    """1-based object ids (B) int64 -> graph selector (B) int32 = obj_ids - 1 (pipeline_lm.py:56-57); ids outside [1, G]
    trap on the device (cp_graph_sel)."""
    _need_cuda(obj_ids)
    ids = obj_ids.contiguous().to(torch.int64)
    out = torch.empty(ids.shape, dtype=torch.int32, device=ids.device)
    check(lib.cp_graph_sel(_p(ids), ids.numel(), int(G), _p(out), _stream()), "cp_graph_sel")
    _count()
    return out


# ------------------------------------------------------------------------------------- K4 decode
def decode_init(logits, L, Ltot, roi_bit, x_bits, y_bits, roi_mask, x_id, y_id, perm=None, graph_sel=None):
    """perm (G,N) int32: plan position -> keypoint id of the logit rows (None = rows already in keypoint order)."""
    _need_cuda(logits, roi_bit, x_bits, y_bits, roi_mask, x_id, y_id, perm, graph_sel)
    B, N = x_id.shape
    check(lib.cp_decode_init(_p(logits), logits.shape[-1], L, Ltot, _p(roi_bit), _p(x_bits), _p(y_bits), _p(roi_mask),
                             _p(x_id), _p(y_id), B, N, _p(perm), _p(graph_sel), _stream()), "cp_decode_init")
    _count()


def decode_refine(logits, plane, Ltot, x_bits, y_bits, x_id, y_id, perm=None, graph_sel=None, x_id_kp=None, y_id_kp=None):
    """x_id_kp / y_id_kp (B,N) int64: also write the updated ids in keypoint order (last stage)."""
    _need_cuda(logits, x_bits, y_bits, x_id, y_id, perm, graph_sel, x_id_kp, y_id_kp)
    B, N = x_id.shape
    check(lib.cp_decode_refine(_p(logits), logits.shape[-1], plane, Ltot, _p(x_bits), _p(y_bits), _p(x_id), _p(y_id),
                               _p(x_id_kp), _p(y_id_kp), B, N, _p(perm), _p(graph_sel), _stream()), "cp_decode_refine")
    _count()


def query_decode_fwd(*, src, w1_packed, b1, slope, w2, b2, plane, Ltot, x_bits, y_bits, x_id, y_id, perm=None, graph_sel=None,
                     x_id_kp=None, y_id_kp=None, logits=None, w_stride=0, b_stride=0):
    """Fused tail of a refine stage (cp_query_decode_fwd): src (B,N,kin) bf16 -> lrelu(Linear kin->64) -> Linear 64->2 -> the
    decode of decode_refine (bit planes, id = 2 id + bit in place, keypoint-order ids).  One launch, TMA tensor loads.
    Object-indexed weights (RoI b uses object graph_sel[b]): ``w_stride`` = (w1_packed bytes, w2 floats), ``b_stride`` = (b1, b2)
    floats between consecutive objects; w2 is then (G, 2, 64)."""
    _need_cuda(src, w1_packed, b1, w2, b2, x_bits, y_bits, x_id, y_id, perm, graph_sel, x_id_kp, y_id_kp, logits)
    assert src.dtype == torch.bfloat16 and src.stride(-1) == 1 and w2.dtype == torch.float32 and w2.is_contiguous() and tuple(w2.shape[-2:]) == (2, 64)
    B, N, kin = src.shape
    p = QueryDecodeParams()
    p.B, p.N = B, N
    p.src, p.ld_src, p.kin = _p(src), src.stride(-2), kin
    p.w1_packed, p.b1, p.nmid, p.slope = _p(w1_packed), _p(b1), 64, float(slope)
    p.w2, p.b2, p.nout = _p(w2), _p(b2), 2
    p.logits, p.ld_logits = _p(logits), (0 if logits is None else logits.shape[-1])
    p.plane, p.Ltot = int(plane), int(Ltot)
    p.x_bits, p.y_bits, p.x_id, p.y_id, p.x_id_kp, p.y_id_kp = _p(x_bits), _p(y_bits), _p(x_id), _p(y_id), _p(x_id_kp), _p(y_id_kp)
    p.perm, p.graph_sel = _p(perm), _p(graph_sel)
    p.w1_stride, p.w2_stride = (0, 0) if w_stride == 0 else (int(w_stride[0]), int(w_stride[1]))
    p.b1_stride, p.b2_stride = (0, 0) if b_stride == 0 else (int(b_stride[0]), int(b_stride[1]))
    _timed_launch(lib.cp_query_decode_fwd, "cp_query_decode_fwd", p, ("QT", kin, (64, 2), OUT_F32, B, N))


def permute_rows(x, perm, graph_sel, to_keypoint_order):
    """x (B,N,...) contiguous -> same shape; rows moved between plan order and keypoint order (cp_permute_rows)."""
    _need_cuda(x, perm, graph_sel)
    x = x.contiguous()
    B, N = x.shape[0], x.shape[1]
    row_bytes = (x.numel() // (B * N)) * x.element_size()
    out = torch.empty_like(x)
    check(lib.cp_permute_rows(_p(x), _p(out), row_bytes, B, N, _p(perm), _p(graph_sel), int(bool(to_keypoint_order)),
                              _stream()), "cp_permute_rows")
    _count()
    return out


CORR_DTYPE_BYTES = 12


def correspondences(roi_bit, seg, bbox, x_id, y_id, out=None):
    """-> (B,N,3) int32 view of records {f32 u, f32 v, u32 flags}; see cp_correspondences."""
    _need_cuda(roi_bit, seg, bbox, x_id, y_id)
    B, N = x_id.shape
    S = seg.shape[-1]
    assert seg.shape[1] == 2 and seg.is_contiguous() and roi_bit.is_contiguous() and bbox.shape == (B, 4)
    if out is None:
        out = torch.empty((B, N, 3), dtype=torch.int32, device=x_id.device)
    check(lib.cp_correspondences(_p(roi_bit), _p(seg.float()), _p(bbox.contiguous().float()), _p(x_id), _p(y_id), _p(out),
                                 B, N, S, _stream()), "cp_correspondences")
    _count()
    return out


def packed_row_bytes(N: int) -> int:
    return 16 + 2 * int(N)


def correspondences_packed(roi_bit, seg, bbox, x_id, y_id, out=None):
    """-> (B, 16 + 2N) uint8 rows {f32 bbox[4]; u16 rec[N]}, rec = x_id | y_id << 6 | flags << 12 (cp_correspondences_pack):
    the payload of the multi-GPU gather and of the device->host read-back, 2 bytes per keypoint."""
    _need_cuda(roi_bit, seg, bbox, x_id, y_id)
    B, N = x_id.shape
    S = seg.shape[-1]
    assert seg.shape[1] == 2 and seg.is_contiguous() and roi_bit.is_contiguous() and bbox.shape == (B, 4)
    if out is None:
        out = torch.empty((B, packed_row_bytes(N)), dtype=torch.uint8, device=x_id.device)
    check(lib.cp_correspondences_pack(_p(roi_bit), _p(seg.float()), _p(bbox.contiguous().float()), _p(x_id), _p(y_id), _p(out),
                                      B, N, S, _stream()), "cp_correspondences_pack")
    _count()
    return out


def unpack_correspondences(packed: torch.Tensor, S: int = 64, out=None):
    """(B, 16 + 2N) uint8 packed rows (CUDA) -> (B,N,3) int32 records, bit-identical to ``correspondences``."""
    _need_cuda(packed)
    assert packed.dtype == torch.uint8 and packed.is_contiguous()
    B = packed.shape[0]
    N = (packed.shape[1] - 16) // 2
    if out is None:
        out = torch.empty((B, N, 3), dtype=torch.int32, device=packed.device)
    check(lib.cp_correspondences_unpack(_p(packed), _p(out), B, N, int(S), _stream()), "cp_correspondences_unpack")
    _count()
    return out


def unpack_correspondences_host(packed, S: int = 64):
    """Host-side consumer of the packed rows (numpy; the PnP stage that reads them runs on the CPU):
    (B, 16 + 2N) uint8 -> (uv (B,N,2) float32, flags (B,N) int32, x_id, y_id (B,N) int32, bbox (B,4) float32)."""
    import numpy as np
    a = np.ascontiguousarray(packed.cpu().numpy() if isinstance(packed, torch.Tensor) else packed)
    bbox = a[:, :16].copy().view(np.float32)
    w = a[:, 16:].copy().view(np.uint16).astype(np.int32)
    x_id, y_id, flags = w & 63, (w >> 6) & 63, w >> 12
    bb = bbox.astype(np.float64)
    u = (bb[:, 2:3] / S) * x_id + bb[:, 0:1]
    v = (bb[:, 3:4] / S) * y_id + bb[:, 1:2]
    return np.stack([u, v], axis=-1).astype(np.float32), flags, x_id, y_id, bbox


FLAG_ALL, FLAG_FULL, FLAG_VISIB = 1, 2, 4


def pnp_ransac(packed, p3d_xyz, cam_K, graph_sel=None, flag=FLAG_ALL, reproj_thresh=2.0, iterations=150, seed=0,
               return_inlier_mask=False, S=64):
    """Batched RANSAC PnP over correspondence records (cp_pnp_ransac): ``packed`` is either the (B, 16 + 2N) uint8 rows of
    ``correspondences_packed`` or the (B,N,3) int32 records of ``correspondences``; p3d_xyz (G,N,3) f32 object keypoints in mm,
    cam_K (3,3) or (B,3,3) -> (R (B,3,3) f32, t (B,3) f32, inlier count (B) int32[, mask (B,N) u8])."""
    _need_cuda(packed, p3d_xyz, cam_K, graph_sel)
    assert packed.is_contiguous()
    B = packed.shape[0]
    is_packed = packed.dtype == torch.uint8
    N = (packed.shape[1] - 16) // 2 if is_packed else packed.shape[1]
    p3d = p3d_xyz.reshape(-1, N, 3).contiguous().float()
    Kc = cam_K.reshape(-1, 9).contiguous().float()
    if Kc.shape[0] not in (1, B):
        raise RuntimeError("pnp_ransac: cam_K must be (3,3) or (B,3,3)")
    pose = torch.empty((B, 12), dtype=torch.float32, device=packed.device)
    ninl = torch.empty((B,), dtype=torch.int32, device=packed.device)
    mask = torch.empty((B, N), dtype=torch.uint8, device=packed.device) if return_inlier_mask else None
    check(lib.cp_pnp_ransac(_p(packed if is_packed else None), _p(None if is_packed else packed), _p(p3d), _p(graph_sel), _p(Kc), int(Kc.shape[0] == B and B > 1), int(flag), float(reproj_thresh),
                            int(iterations), int(seed) & 0xFFFFFFFFFFFFFFFF, _p(pose), _p(ninl), _p(mask), B, N, int(S), _stream()),
          "cp_pnp_ransac")
    _count()
    R, t = pose[:, :9].reshape(B, 3, 3), pose[:, 9:]
    return (R, t, ninl, mask) if return_inlier_mask else (R, t, ninl)


def split_correspondences(rec: torch.Tensor):
    """(…,3) int32 records -> (uv float32 (…,2), flags int32 (…))."""
    uv = rec[..., :2].contiguous().view(torch.float32)
    return uv, rec[..., 2]


def threshold(x, thr=0.5, apply_sigmoid=True, as_long=False):
    _need_cuda(x)
    x = x.contiguous().float()
    out = torch.empty(x.shape, dtype=torch.int64 if as_long else torch.float32, device=x.device)
    check(lib.cp_threshold(_p(x), float(thr), int(apply_sigmoid), _p(out), int(as_long), x.numel(), _stream()), "cp_threshold")
    _count()
    return out


def bits_to_id(x, code_dim, binarize, thr=0.5, base=2, as_long=True):
    """Reduce dimension ``code_dim`` of x (MSB first) to an id; output has that dimension removed."""
    _need_cuda(x)
    x = x.contiguous().float()
    shape = list(x.shape)
    L = shape[code_dim]
    outer = 1
    for s in shape[:code_dim]:
        outer *= s
    inner = 1
    for s in shape[code_dim + 1:]:
        inner *= s
    out_shape = shape[:code_dim] + shape[code_dim + 1:]
    out = torch.empty(out_shape, dtype=torch.int64 if as_long else torch.float32, device=x.device)
    check(lib.cp_bits_to_id(_p(x), outer, L, inner, L * inner, inner, 1, int(binarize), float(thr), int(base), _p(out),
                            int(as_long), _stream()), "cp_bits_to_id")
    _count()
    return out


def id_to_bits(ids, L, base=2):
    """ids (...,) int64 -> (..., L) f32 digits, MSB first (class_id_encoder_decoder.py:88-101)."""
    _need_cuda(ids)
    ids = ids.contiguous().to(torch.int64)
    out = torch.empty(tuple(ids.shape) + (int(L),), dtype=torch.float32, device=ids.device)
    check(lib.cp_id_to_bits(_p(ids), ids.numel(), int(L), int(base), _p(out), _stream()), "cp_id_to_bits")
    _count()
    return out


def group_argmax(x, D):
    """x (G*D, H, W)-like viewed as (G, D, inner) -> (G, inner) int64 argmax over D."""
    _need_cuda(x)
    x = x.contiguous().float()
    total = x.numel()
    inner = 1
    for s in x.shape[2:]:
        inner *= s
    G = total // (D * inner)
    out = torch.empty((G, inner), dtype=torch.int64, device=x.device)
    check(lib.cp_group_argmax(_p(x), G, int(D), inner, _p(out), _stream()), "cp_group_argmax")
    _count()
    return out
