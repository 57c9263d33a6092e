"""Drop-in for checkerpose/model/pipeline_lm.py (LM-13 multi-object nets): identical maths, but
``knn_idx`` is a (num_obj, N, K) table and every EdgeConv selects its graph per sample with the
1-based ``obj_ids`` (pipeline_lm.py:55-57) -- the kernels take that as a per-RoI graph selector."""
import torch
import torch.nn as nn

from .. import head, ops
from .pipeline import (IMG_FEATS_DIMS, Index2Feat_module, MLP_QueryNet, from_bit_prob_to_id,  # noqa: F401
                       from_code_prob_to_id, from_code_to_id, from_gt_bit_to_id, from_gt_code_to_id,
                       from_mask_prob_to_mask, get_gdrn_upsample_module, get_graph_feature,
                       get_MLP_leakyReLU_layers, knn, _to_io)
from . import pipeline as _single


class StaticGraph_module(_single.StaticGraph_module):
    def forward(self, x, batch_indices, obj_ids):
        return self._forward_impl(x, obj_ids)


class Refine_moduleGNN(_single.Refine_moduleGNN):
    _graph_module_cls = StaticGraph_module

    def forward(self, img_feat, graph_feat, p3d_normed, roi_mask_bit, prev_x_id, prev_y_id, obj_ids):
        return self._forward_impl(img_feat, graph_feat, roi_mask_bit, prev_x_id, prev_y_id, obj_ids)


class PoseNet_GNNskip(_single.PoseNet_GNNskip):
    _refine_cls = Refine_moduleGNN

    def forward(self, img, p3d_normed, obj_ids, stage=None):
        img_feats = self.init_net.img_backbone(img)
        out, _ = head.pose_head_forward(self, img_feats, obj_ids=obj_ids, stage=stage)
        return out


class Refine_moduleGNN_ABwoProg(head.DeviceScopedModule):
    """Ablation stage without progressive refinement (pipeline_lm.py:286-339): Linear+LeakyReLU x2 on the graph
    feature, then ``num_graph_module`` EdgeConv layers; no image sampling, no per-stage query."""

    def __init__(self, npoint, p3d_normed, num_filters=256, max_batch_size=64, query_dims=None,
                 local_k=4, leaky_slope=0.01, num_graph_module=2, graph_k=20, graph_leaky_slope=0.2,
                 query_type="mlp", graph_feat_dim=64):
        super(Refine_moduleGNN_ABwoProg, self).__init__()
        self.npoint = npoint
        if query_type == "mlp":
            self.query_dims = (num_filters, 256, 64) if query_dims is None else tuple(query_dims)
        else:
            raise ValueError("query type {} not supported in Refine_module".format(query_type))
        self.max_batch_size = max_batch_size  # kept for API compatibility; no index tables are allocated
        self.pre_graph_module = get_MLP_leakyReLU_layers(dims=(graph_feat_dim, self.query_dims[0], self.query_dims[0]),
                                                         doLastAct=True, negative_slope=leaky_slope)
        self.pre_query_block = nn.ModuleList()
        knn_idx = _single.LazyKnnGraph(p3d_normed, graph_k)
        for i in range(num_graph_module):
            self.pre_query_block.append(StaticGraph_module(input_dim=self.query_dims[0], output_dim=self.query_dims[0],
                                                           knn_idx=knn_idx, leaky_slope=graph_leaky_slope))

    def forward(self, graph_feat, obj_ids):
        dtype = head.get_compute_dtype()
        B = graph_feat.shape[0]
        blocks = list(self.pre_query_block)
        ctx = head.graph_ctx(blocks[0]._knn, obj_ids, B, graph_feat.device) if blocks else None
        gfeat = ops.to_node_major(graph_feat, dtype)
        if ctx is not None:
            gfeat = ctx.to_plan(gfeat)
        feat = head.abwoprog_refine_node_major(self, gfeat, ctx, dtype)[:, :, :self.query_dims[0]]   # bf16: width padded
        if ctx is not None:
            feat = ctx.to_keypoints(feat)
        return _to_io(feat, graph_feat.dtype)


class PoseNet_GNNskip_ABwoProg(head.DeviceScopedModule):
    """Ablation net without progressive refinement (pipeline_lm.py:430-517): the stages refine the graph feature
    only; ONE MLP_QueryNet emits all 2*res_log2+1 logits at the end.  Same constructor, ``forward`` signature, return
    tuple and state_dict keys as the reference."""

    def __init__(self, init_net, npoint, p3d_normed, res_log2=6, num_filters=256, max_batch_size=64, query_dims=None,
                 seg_output_dim=2, local_k=4, leaky_slope=0.01, num_graph_module=2, graph_k=20, graph_leaky_slope=0.2,
                 query_type="mlp"):
        super(PoseNet_GNNskip_ABwoProg, self).__init__()
        self.npoint = npoint
        self.init_net = init_net
        self.res_log2 = res_log2
        self.num_bits = 2 * res_log2 + 1
        self.num_refine_steps = res_log2 - 3
        self.up_net = nn.ModuleList()
        for i in range(self.num_refine_steps):
            if i == 0:
                block = get_gdrn_upsample_module(is_convtrans=True, in_channels=IMG_FEATS_DIMS[self.init_net.backbone_name][-1],
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
            self.refine_net.append(Refine_moduleGNN_ABwoProg(
                npoint=npoint, p3d_normed=p3d_normed, num_filters=num_filters, max_batch_size=max_batch_size,
                query_dims=query_dims, local_k=local_k, leaky_slope=leaky_slope, num_graph_module=num_graph_module_i,
                graph_k=graph_k, graph_leaky_slope=graph_leaky_slope, query_type=query_type, graph_feat_dim=graph_feat_dim_i))
        self.seg_block = nn.Conv2d(num_filters, seg_output_dim, kernel_size=1, padding=0, bias=True)
        if query_type == "mlp":
            self.query_dims = (num_filters, 256, 64) if query_dims is None else tuple(query_dims)
            self.query_block = MLP_QueryNet(feat_dims=self.query_dims, pt_dim=3, out_dim=self.num_bits, leaky_slope=leaky_slope)
        else:
            raise ValueError("query type {} not supported in Refine_module".format(query_type))

    def forward(self, img, p3d_normed, obj_ids, stage=None):
        img_feats = self.init_net.img_backbone(img)
        return head.abwoprog_head_forward(self, img_feats, obj_ids, stage=stage)
