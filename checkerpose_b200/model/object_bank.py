"""One head forward over a batch of RoIs of many objects, each object with its own PoseNet_GNNskip.

CheckerPose trains one network per object (8 on LM-O, 21 on YCB-V), each with its own checkpoint and FPS keypoints, while a
detector hands the head RoIs of many objects at once.  ``ObjectBank`` serves such a batch:

* the RoIs are stably sorted by object (the order only changes where work runs; outputs come back in the caller's order);
* the image branch (backbone, ``up_net``, ``patch_generator``, ``seg_block``, ``conv1x1``) runs per object group, with the
  group's own net, on the group's contiguous rows of the sorted batch;
* bf16 mode: everything from the first EdgeConv to the decode runs as ONE launch per layer over the whole sorted batch, each
  tile with its object's weights (the kernels' object-indexed weights, selected by the per-RoI graph selector) and its
  object's kNN graph;
* float32 mode runs every object group through its own net's float32 path.

Results equal, bit for bit, what each object's own net computes on its RoIs.  The group sizes are needed on the host: ids
given on the GPU are copied to the host once per forward (the forward's only synchronisation), and an id that is not a key
of the bank raises there in either case.
"""
from __future__ import annotations

from typing import Mapping

import numpy as np
import torch
import torch.nn as nn

from .. import head, ops


def _same(field, vals):
    if any(v != vals[0] for v in vals[1:]):
        raise ValueError(f"ObjectBank members differ in {field}: {vals}")


def _arch_fields(net):
    """What the batched kernels need all members to share, field by field."""
    inet, ref0 = net.init_net, net.refine_net[0]
    qmods = [ref0.query_block.mlps[i] for i in (0, 2, 4)]
    return {
        "npoint": net.npoint,
        "graph_k": inet.pre_query_block[0]._knn.k if inet.pre_query_block and hasattr(inet.pre_query_block[0]._knn, "k") else None,
        "res_log2": net.num_refine_steps + 3,
        "query_dims": tuple(ref0.query_dims),
        "num_filters": ref0.local_feat_ext_block.patch_generator.in_channels,
        "num_graph_module": tuple(len(r.pre_query_block) for r in net.refine_net),
        "init num_graph_module": len(inet.pre_query_block),
        "local_k": ref0.local_feat_ext_block.kernel_size,
        "slopes": (float(ref0.pre_graph_module[1].negative_slope), float(ref0.query_block.mlps[1].negative_slope),
                   tuple(float(b.conv[2].negative_slope) for r in [inet] + list(net.refine_net) for b in r.pre_query_block)),
        "backbone feature dims": (inet.backbone_name, inet.conv1x1.in_channels if isinstance(inet.conv1x1, nn.Conv2d) else None,
                                  tuple(m.in_channels for blk in net.up_net for m in blk if isinstance(m, (nn.Conv2d, nn.ConvTranspose2d)))),
        "query MLP": tuple(tuple(m.weight.shape) for m in qmods),
    }


def _take(img, idx):
    """Rows ``idx`` of the batch: a tensor, or a list / tuple of per-level tensors (a FeatureListBackbone input)."""
    if isinstance(img, (list, tuple)):
        return type(img)(t.index_select(0, idx) for t in img)
    return img.index_select(0, idx)


def _rows(img, s, e):
    if isinstance(img, (list, tuple)):
        return type(img)(t[s:e] for t in img)
    return img[s:e]


def _device(img):
    return (img[0] if isinstance(img, (list, tuple)) else img).device


class ObjectBank(head.DeviceScopedModule):
    """``nets``: 1-based object id -> that object's PoseNet_GNNskip (one architecture, own weights and keypoints)."""

    def __init__(self, nets: Mapping[int, nn.Module]):
        super().__init__()
        if not nets:
            raise ValueError("ObjectBank needs at least one net")
        self.obj_keys = sorted(int(k) for k in nets)
        self.nets = nn.ModuleList([nets[k] for k in sorted(nets)])
        fields = [_arch_fields(n) for n in self.nets]
        for f in fields[0]:
            _same(f, [fl[f] for fl in fields])
        if fields[0]["init num_graph_module"] == 0 or 0 in fields[0]["num_graph_module"]:
            raise ValueError("ObjectBank members need graph modules in the init net and in every refine stage")
        self._index = {k: i for i, k in enumerate(self.obj_keys)}
        self._engine = head.BankEngine(list(self.nets))
        self.training = any(n.training for n in self.nets)     # a bank of eval() nets starts in eval mode

    def _order(self, obj_ids, B):
        ids = np.asarray(obj_ids.detach().cpu() if isinstance(obj_ids, torch.Tensor) else obj_ids).reshape(-1)
        if ids.shape[0] != B:
            raise ValueError(f"obj_ids has {ids.shape[0]} entries for a batch of {B}")
        bad = sorted({int(i) for i in ids} - set(self._index))
        if bad:
            raise ValueError(f"object ids {bad} are not in the bank (keys {self.obj_keys})")
        g = np.array([self._index[int(i)] for i in ids], dtype=np.int64)
        order = np.argsort(g, kind="stable")
        gs = g[order]
        starts = np.flatnonzero(np.r_[True, gs[1:] != gs[:-1]])
        ends = np.r_[starts[1:], B]
        return g, order, [(int(gs[s]), int(s), int(e)) for s, e in zip(starts, ends)]

    def _head(self, img, obj_ids, stage, bbox, packed):
        head._require_eval(self)
        dev = _device(img)
        B = (img[0] if isinstance(img, (list, tuple)) else img).shape[0]
        g, order, groups = self._order(obj_ids, B)
        in_order = bool((order == np.arange(B)).all())         # already grouped: no copy of the inputs
        perm = torch.from_numpy(order).to(dev)
        inv = torch.from_numpy(np.argsort(order)).to(dev)
        img_s = img if in_order else _take(img, perm)
        bbox_s = None if bbox is None or in_order else bbox.index_select(0, perm)
        bbox_s = bbox if in_order else bbox_s
        feats = [self.nets[gi].init_net.img_backbone(_rows(img_s, s, e)) for gi, s, e in groups]
        dtype = head.get_compute_dtype()
        with torch.cuda.device(dev):
            if dtype == torch.float32:
                res = [head.pose_head_forward(self.nets[gi], f, None, stage, dtype, None if bbox_s is None else bbox_s[s:e], packed)
                       for (gi, s, e), f in zip(groups, feats)]
                out = tuple(torch.cat([r[0][k] for r in res]) for k in range(6))
                corr = None if bbox is None else torch.cat([r[1] for r in res])
            else:
                if head.get_image_branch() != "tcgen05":
                    raise RuntimeError("ObjectBank runs the bf16 head with the tcgen05 image branch")
                img_feats = [head.GroupMaps([f[lvl] for f in feats], groups) for lvl in range(len(feats[0]))]
                sel_ids = torch.from_numpy(g[order] + 1).to(dev)       # 1-based bank index of every sorted RoI
                with head.object_bank(self._engine):
                    out, corr = head.pose_head_forward(self.nets[0], img_feats, obj_ids=sel_ids, stage=stage, dtype=dtype,
                                                       bbox=bbox_s, packed=packed)
            if not in_order:
                out = tuple(t.index_select(0, inv) for t in out)
                corr = None if corr is None else corr.index_select(0, inv)
        return out, corr, g

    def forward(self, img, obj_ids, stage=None):
        """-> the reference's 6-tuple (roi_bit, x_bits, y_bits, seg, x_id, y_id) for every RoI, in the caller's order."""
        return self._head(img, obj_ids, stage, None, False)[0]

    def forward_with_correspondences(self, img, bbox, obj_ids, stage=None, packed=False):
        """-> (6-tuple, correspondence records): PoseNet_GNNskip.forward_with_correspondences for a mixed batch."""
        out, corr, _ = self._head(img, obj_ids, stage, bbox, packed)
        return out, corr

    def forward_with_pose(self, img, bbox, p3d_xyz, cam_K, obj_ids, stage=None, flag=ops.FLAG_ALL, reproj_thresh=2.0,
                          iterations=150, seed=0):
        """PoseNet_GNNskip.forward_with_pose for a mixed batch: p3d_xyz (G,N,3) keypoints in mm of the bank's objects in key
        order, cam_K (3,3) or (B,3,3).  -> (6-tuple, packed records, R (B,3,3), t (B,3), inlier counts (B)).  PnP runs once per
        object group, so that every RoI draws the hypotheses it draws in its own net's batch."""
        out, packed, g = self._head(img, obj_ids, stage, bbox, True)
        dev = packed.device
        B, N = packed.shape[0], self.nets[0].npoint
        p3d = p3d_xyz.reshape(-1, N, 3)
        if p3d.shape[0] != len(self.obj_keys):
            raise ValueError(f"p3d_xyz holds {p3d.shape[0]} objects, the bank {len(self.obj_keys)}")
        K = cam_K.reshape(-1, 3, 3)
        R = torch.empty((B, 3, 3), dtype=torch.float32, device=dev)
        t = torch.empty((B, 3), dtype=torch.float32, device=dev)
        ninl = torch.empty((B,), dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            for gi in np.unique(g):
                rows = torch.from_numpy(np.flatnonzero(g == gi)).to(dev)
                Kg = cam_K if K.shape[0] == 1 else K.index_select(0, rows)
                Rg, tg, ng = ops.pnp_ransac(packed.index_select(0, rows), p3d[gi:gi + 1], Kg, flag=flag, reproj_thresh=reproj_thresh,
                                            iterations=iterations, seed=seed)
                R[rows], t[rows], ninl[rows] = Rg, tg, ng
        return out, packed, R, t, ninl
