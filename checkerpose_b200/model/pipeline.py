"""Drop-in for checkerpose/model/pipeline.py -- same names, signatures, state_dict keys and return
values; every op on the GNN path runs on the hand-written sm_100a kernels (no CPU fallback).

Differences that are deliberate and invisible to callers:
* ``max_batch_size`` is accepted but the (max_B, N*K) int64 ``pre_batch_indices`` / ``batch_indices``
  tables of the reference (pipeline.py:235-252; 671 MB each at max_B=1024, N=4096) are never built;
  the ``batch_indices`` arguments of the forward methods are accepted and ignored.
* modules are inference-only (BatchNorm is folded): calling them in training mode raises.
* (B,C,N) results are permuted views of node-major (B,N,C) storage, exactly like the reference's own
  ``output_feat`` (pipeline.py:297).
"""
import torch
import torch.nn as nn

from .. import head, ops

IMG_FEATS_DIMS = {
    "resnet34": [64, 128, 256, 512],
    "convnext_tiny": [192, 384, 768],
    "convnext_small": [192, 384, 768],
    "convnext_base": [256, 512, 1024],
    "darknet53": [64, 128, 256, 512, 1024],
    "hrnet_w18": [128, 256, 512, 1024],
    "hrnet_w18_small": [128, 256, 512, 1024],
    "hrnet_w30": [128, 256, 512, 1024],
}


def knn(x, k):
    """x (B,C,N) -> idx (B,N,k) int64.  pipeline.py:18-23 (kernel K1)."""
    return ops.knn(x, k)


class LazyKnnGraph:
    """The static graph ``knn(p3d_normed, graph_k)`` the reference builds in ``__init__``
    (pipeline.py:248, init.py:98).  Built immediately when the keypoints already live on a GPU (the
    reference's behaviour); when a net is constructed on the CPU and moved with ``.cuda()`` later, the
    graph is built on first use -- there is no CPU kNN."""

    def __init__(self, p3d_normed, k):
        self.p3d_normed, self.k, self._idx = p3d_normed, int(k), None
        if p3d_normed.is_cuda:
            self._idx = ops.knn(p3d_normed, self.k)

    def get(self, device=None):
        dev = None if device is None else torch.device(device)
        stale = self._idx is None or (dev is not None and dev.type == "cuda" and dev.index is not None
                                      and dev.index != self._idx.device.index)
        if stale:
            if dev is None or dev.type != "cuda":
                raise RuntimeError("the kNN graph is built by a CUDA kernel: move the keypoints or the net to a GPU first")
            with torch.cuda.device(dev):
                self._idx = ops.knn(self.p3d_normed.to(dev), self.k)
        return self._idx


def get_graph_feature(x, knn_idx, batch_indices=None):
    """x (B,C,N), knn_idx (1|B,N,K) -> (B,2C,N,K).  pipeline.py:27-40 (API completeness only)."""
    idx32, sel = head.graph_select(knn_idx, None, x.shape[0], x.device)
    return ops.graph_feature(x, idx32, sel)


def _to_io(x_nm, like_dtype):
    """node-major result -> (B,C,N) view in the caller's dtype."""
    return ops.convert(x_nm, like_dtype).permute(0, 2, 1)


class StaticGraph_module(head.DeviceScopedModule):
    """EdgeConv with a fixed kNN graph (pipeline.py:45-59): kernel K2."""

    def __init__(self, input_dim, output_dim, knn_idx, leaky_slope=0.2):
        super(StaticGraph_module, self).__init__()
        self._knn = knn_idx  # tensor (1|G,N,K) int64 as in the reference, or a LazyKnnGraph
        self.conv = nn.Sequential(
            nn.Conv2d(input_dim * 2, output_dim, kernel_size=1, bias=False),
            nn.BatchNorm2d(output_dim),
            nn.LeakyReLU(negative_slope=leaky_slope)
        )

    @property
    def knn_idx(self):
        return self._knn.get() if isinstance(self._knn, LazyKnnGraph) else self._knn

    @knn_idx.setter
    def knn_idx(self, value):
        self._knn = value

    def _forward_impl(self, x, obj_ids):
        dtype = head.get_compute_dtype()
        ctx = head.graph_ctx(self._knn, obj_ids, x.shape[0], x.device)
        y = head.edgeconv_node_major(self, ctx.to_plan(ops.to_node_major(x, dtype)), ctx, dtype)
        y = y[:, :, :self.conv[0].weight.shape[0]]     # bf16 mode keeps the width padded to a multiple of 64
        return _to_io(ctx.to_keypoints(y), x.dtype)

    def forward(self, x, batch_indices=None):
        return self._forward_impl(x, None)


def get_MLP_leakyReLU_layers(dims, doLastAct, negative_slope=0.1):
    layers = []
    for i in range(1, len(dims)):
        layers.append(nn.Linear(dims[i - 1], dims[i]))
        if i == len(dims) - 1 and not doLastAct:
            continue
        layers.append(nn.LeakyReLU(negative_slope=negative_slope))
    return nn.Sequential(*layers)


def from_code_to_id(code, class_base=2):
    """(B,L,N) integer code -> (B,N) ids, MSB first.  pipeline.py:72-82."""
    return ops.bits_to_id(code, 1, binarize=False, base=class_base, as_long=True)


def from_code_prob_to_id(code_prob, class_base=2):
    """(B,L,N) logits -> ids; bit = sigmoid(x) > 0.5.  pipeline.py:84-92."""
    return ops.bits_to_id(code_prob, 1, binarize=True, thr=0.0, base=class_base, as_long=True)


def from_gt_code_to_id(gt_code, class_base=2):
    return ops.bits_to_id(gt_code, 1, binarize=True, thr=0.5, base=class_base, as_long=True)  # pipeline.py:94-101


def from_bit_prob_to_id(bit_prob):
    return ops.threshold(bit_prob[:, 0, :], thr=0.0, apply_sigmoid=False, as_long=True)  # pipeline.py:103-110


def from_gt_bit_to_id(gt_bit):
    return ops.threshold(gt_bit[:, 0, :], thr=0.5, apply_sigmoid=False, as_long=True)  # pipeline.py:112-118


def from_mask_prob_to_mask(mask_prob):
    return ops.threshold(mask_prob, thr=0.0, apply_sigmoid=False, as_long=False)  # pipeline.py:120-127


class Index2Feat_module(head.DeviceScopedModule):
    """Patch embedding conv + exact 4-tap integer gather (pipeline.py:130-164): kernel K3."""

    def __init__(self, feat_dim, embed_dim=None, kernel_size=2):
        super(Index2Feat_module, self).__init__()
        self.kernel_size = kernel_size
        self.embed_dim = embed_dim if embed_dim is not None else (feat_dim * kernel_size * kernel_size)
        self.patch_generator = nn.Conv2d(in_channels=feat_dim, out_channels=self.embed_dim,
                                         kernel_size=kernel_size, stride=1, padding=kernel_size - 1)

    def forward(self, img_feat_highres, batch_indices, pixel_x_id, pixel_y_id):
        dtype = head.get_compute_dtype()
        patches = head.patches_nhwc(self.patch_generator, img_feat_highres, dtype)
        out = ops.sample_taps(patches, pixel_x_id.contiguous(), pixel_y_id.contiguous(), None, self.kernel_size)
        return _to_io(out, img_feat_highres.dtype)


class MLP_QueryNet(head.DeviceScopedModule):
    """Linear stack on (B,N,C) tensors; ``pts`` is unused, as in the reference (pipeline.py:168-180)."""

    def __init__(self, feat_dims=(256, 256, 64), pt_dim=3, out_dim=4, leaky_slope=0.01):
        super(MLP_QueryNet, self).__init__()
        mlp_dims = tuple(feat_dims) + (out_dim,)
        self.mlps = get_MLP_leakyReLU_layers(dims=mlp_dims, doLastAct=False, negative_slope=leaky_slope)

    def forward(self, img_feats, pts=None):
        # standalone use runs the exact fp32 GEMM; inside Refine_moduleGNN the bf16 mode fuses these layers
        if not img_feats.is_cuda:
            raise RuntimeError("checkerpose_b200: expected a CUDA tensor (there is no CPU fallback)")
        x = img_feats.float()
        mods = list(self.mlps)
        i = 0
        while i < len(mods):
            lin = head.prepared_linear(mods[i], torch.float32)
            act = i + 1 < len(mods) and isinstance(mods[i + 1], nn.LeakyReLU)
            x = ops.linear_f32(x, lin.w, lin.b, act, mods[i + 1].negative_slope if act else 0.0)
            i += 2 if act else 1
        return x.to(img_feats.dtype)


def get_gdrn_upsample_module(is_convtrans=False, in_channels=512, num_filters=256, kernel_size=3, padding=1,
                             output_padding=1):
    """Image-branch block (pipeline.py:183-211); dense convolution, runs on cuDNN."""
    layers = []
    if is_convtrans:
        layers.append(nn.ConvTranspose2d(in_channels, num_filters, kernel_size=kernel_size, stride=2, padding=padding,
                                         output_padding=output_padding, bias=False))
        layers.append(nn.BatchNorm2d(num_features=num_filters))
        layers.append(nn.ReLU(inplace=True))
        layers.append(nn.Conv2d(num_filters, num_filters, kernel_size=3, stride=1, padding=1, bias=False))
    else:
        layers.append(nn.UpsamplingBilinear2d(scale_factor=2))
        layers.append(nn.Conv2d(in_channels, num_filters, kernel_size=3, stride=1, padding=1, bias=False))
    layers.append(nn.BatchNorm2d(num_features=num_filters))
    layers.append(nn.ReLU(inplace=True))
    layers.append(nn.Conv2d(num_filters, num_filters, kernel_size=3, stride=1, padding=1, bias=False))
    layers.append(nn.BatchNorm2d(num_features=num_filters))
    layers.append(nn.ReLU(inplace=True))
    return nn.Sequential(*layers)


class Refine_moduleGNN(head.DeviceScopedModule):
    """One refine stage (pipeline.py:214-298): Index2Feat gather -> x roi mask -> cat graph feature ->
    MLP -> num_graph_module x EdgeConv -> MLP_QueryNet."""

    _graph_module_cls = None  # set below (LM variant overrides)

    def __init__(self, npoint, p3d_normed, num_filters=256, max_batch_size=64, query_dims=None,
                 local_k=4, leaky_slope=0.01, num_graph_module=2, graph_k=20, graph_leaky_slope=0.2,
                 query_type="mlp", graph_feat_dim=64):
        super(Refine_moduleGNN, self).__init__()
        self.npoint = npoint
        if query_type == "mlp":
            self.query_dims = (num_filters, 256, 64) if query_dims is None else tuple(query_dims)
        else:
            raise ValueError("query type {} not supported in Refine_module".format(query_type))
        self.max_batch_size = max_batch_size  # kept for API compatibility; no index tables are allocated
        self.local_feat_ext_block = Index2Feat_module(feat_dim=num_filters, embed_dim=self.query_dims[0] // 4,
                                                      kernel_size=local_k)
        self.pre_graph_module = get_MLP_leakyReLU_layers(
            dims=(self.query_dims[0] + graph_feat_dim, self.query_dims[0], self.query_dims[0]),
            doLastAct=True, negative_slope=leaky_slope)
        self.pre_query_block = nn.ModuleList()
        knn_idx = LazyKnnGraph(p3d_normed, graph_k)
        for i in range(num_graph_module):
            self.pre_query_block.append(self._graph_module_cls(input_dim=self.query_dims[0], output_dim=self.query_dims[0],
                                                               knn_idx=knn_idx, leaky_slope=graph_leaky_slope))
        if query_type == "mlp":
            self.query_block = MLP_QueryNet(feat_dims=self.query_dims, pt_dim=3, out_dim=2, leaky_slope=leaky_slope)

    def _forward_impl(self, img_feat, graph_feat, roi_mask_bit, prev_x_id, prev_y_id, obj_ids):
        dtype = head.get_compute_dtype()
        B, N = img_feat.shape[0], self.npoint
        blocks = list(self.pre_query_block)
        ctx = head.graph_ctx(blocks[0]._knn, obj_ids, B, img_feat.device) if blocks else None
        mask = roi_mask_bit.detach().reshape(B, N, 1).contiguous().float()
        gfeat = ops.to_node_major(graph_feat, dtype)
        x_id, y_id = prev_x_id.reshape(B, N, 1).contiguous(), prev_y_id.reshape(B, N, 1).contiguous()
        if ctx is not None:   # the kernels work in the graph plan's node order; the API is in keypoint order
            mask, gfeat, x_id, y_id = ctx.to_plan(mask), ctx.to_plan(gfeat), ctx.to_plan(x_id), ctx.to_plan(y_id)
        logits, feat = head.refine_node_major(self, img_feat, gfeat, mask.view(B, N), x_id.view(B, N), y_id.view(B, N),
                                              ctx, dtype)
        logits = logits[:, :, :2].contiguous()
        feat = feat[:, :, :self.query_dims[0]]          # bf16 mode keeps the width padded to a multiple of 64
        if ctx is not None:
            logits, feat = ctx.to_keypoints(logits), ctx.to_keypoints(feat)
        return logits.permute(0, 2, 1), _to_io(feat, graph_feat.dtype)

    def forward(self, img_feat, graph_feat, p3d_normed, roi_mask_bit, prev_x_id, prev_y_id):
        return self._forward_impl(img_feat, graph_feat, roi_mask_bit, prev_x_id, prev_y_id, None)


Refine_moduleGNN._graph_module_cls = StaticGraph_module


class PoseNet_GNNskip(head.DeviceScopedModule):
    """Full progressive head (pipeline.py:301-384).  ``forward`` returns the reference's 6-tuple."""

    _refine_cls = Refine_moduleGNN

    def __init__(self, init_net, npoint, p3d_normed, res_log2=6, num_filters=256, max_batch_size=64, query_dims=None,
                 seg_output_dim=2, local_k=4, leaky_slope=0.01, num_graph_module=2, graph_k=20, graph_leaky_slope=0.2,
                 query_type="mlp"):
        super(PoseNet_GNNskip, self).__init__()
        self.npoint = npoint
        self.init_net = init_net
        self.num_refine_steps = res_log2 - 3
        self.up_net = nn.ModuleList()
        for i in range(self.num_refine_steps):
            if i == 0:
                block = get_gdrn_upsample_module(is_convtrans=True,
                                                 in_channels=IMG_FEATS_DIMS[self.init_net.backbone_name][-1],
                                                 num_filters=num_filters)
            else:
                block = get_gdrn_upsample_module(is_convtrans=False,
                                                 in_channels=num_filters + IMG_FEATS_DIMS[self.init_net.backbone_name][-i - 1],
                                                 num_filters=num_filters)
            self.up_net.append(block)
        self.refine_net = nn.ModuleList()
        for i in range(self.num_refine_steps):
            num_graph_module_i = num_graph_module if isinstance(num_graph_module, int) else num_graph_module[i]
            if i == 0:
                graph_feat_dim_i = 64
            elif query_dims is None:
                graph_feat_dim_i = num_filters
            else:
                graph_feat_dim_i = query_dims[0]
            self.refine_net.append(self._refine_cls(
                npoint=npoint, p3d_normed=p3d_normed, num_filters=num_filters, max_batch_size=max_batch_size,
                query_dims=query_dims, local_k=local_k, leaky_slope=leaky_slope, num_graph_module=num_graph_module_i,
                graph_k=graph_k, graph_leaky_slope=graph_leaky_slope, query_type=query_type,
                graph_feat_dim=graph_feat_dim_i))
        self.seg_block = nn.Conv2d(num_filters, seg_output_dim, kernel_size=1, padding=0, bias=True)

    def forward_with_correspondences(self, img, p3d_normed, bbox, stage=None, obj_ids=None, packed=False):
        """Extension: the reference's 6-tuple plus (B,N,3) int32 correspondence records
        {f32 u, f32 v, u32 flags} (first half of from_id_to_pose, test_network_with_test_data.py:50-66);
        ``packed``: the 2-byte-per-keypoint rows of ops.correspondences_packed instead."""
        img_feats = self.init_net.img_backbone(img)
        with torch.cuda.device(img_feats[-1].device):
            return head.pose_head_forward(self, img_feats, obj_ids=obj_ids, stage=stage, bbox=bbox, packed=packed)

    def forward_with_pose(self, img, p3d_normed, bbox, p3d_xyz, cam_K, stage=None, obj_ids=None, flag=ops.FLAG_ALL,
                          reproj_thresh=2.0, iterations=150, seed=0):
        """Extension: head + PnP front-end in one call (from_id_to_pose of test_network_with_test_data.py:32-119 for the whole
        batch on the device).  p3d_xyz (G,N,3) object keypoints in mm (G = 1 or one cloud per graph, selected like the kNN
        graphs), cam_K (3,3) or (B,3,3).  -> (the reference's 6-tuple, packed records, R (B,3,3), t (B,3), inlier counts (B)).
        ``flag``: one validity set (ops.FLAG_*) or a tuple of up to 3, solved in one launch; for a tuple R, t and the counts
        gain a leading set axis (V,B,...), entry v equal to the call with flag[v].  ``flag=(ops.FLAG_ALL, ops.FLAG_FULL,
        ops.FLAG_VISIB)`` gives the three poses test.py:335-368 reports (all / full mask / visible mask)."""
        out, packed = self.forward_with_correspondences(img, p3d_normed, bbox, stage=stage, obj_ids=obj_ids, packed=True)
        with torch.cuda.device(packed.device):
            sel = None if obj_ids is None else ops.graph_sel(obj_ids.to(packed.device), p3d_xyz.reshape(-1, self.npoint, 3).shape[0])
            R, t, ninl = ops.pnp_ransac(packed, p3d_xyz, cam_K, graph_sel=sel, flag=flag, reproj_thresh=reproj_thresh,
                                        iterations=iterations, seed=seed)
        return out, packed, R, t, ninl

    def forward(self, img, p3d_normed, stage=None):
        img_feats = self.init_net.img_backbone(img)
        out, _ = head.pose_head_forward(self, img_feats, obj_ids=None, stage=stage)
        return out
