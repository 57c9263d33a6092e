"""ObjectBank host side without a GPU: member checks, id validation, and the ctypes mirrors of the structs that gained
object-indexed weight strides (checked against the header with a C program built by the host compiler)."""
import ctypes as C
import os
import shutil
import subprocess

import pytest
import torch

from helpers import REPO, syn


def _net(N=64, seed=0, dims=None, local_k=2, graph_k=20, obj=1):
    from checkerpose_b200.model import init, pipeline
    from checkerpose_b200.model.backbone import FeatureListBackbone
    p3d = syn.p3d_normed_tensor(syn.load_fps_xyz("lmo", obj, N))
    inet = init.InitNet_GNN(npoint=N, p3d_normed=p3d, res_log2=3, backbone_name="hrnet_w18", pretrain_backbone=False,
                            graph_k=graph_k, img_backbone=FeatureListBackbone())
    net = pipeline.PoseNet_GNNskip(inet, npoint=N, p3d_normed=p3d, res_log2=6, local_k=local_k, num_graph_module=3,
                                   graph_k=graph_k, query_dims=dims)
    return net.eval()


@pytest.mark.parametrize("kw, field", [(dict(N=128), "npoint"), (dict(graph_k=16), "graph_k"), (dict(local_k=4), "local_k"),
                                       (dict(dims=(256, 128, 64)), "query_dims")])
def test_mismatched_members_raise_and_name_the_field(kw, field):
    from checkerpose_b200.model.object_bank import ObjectBank
    with pytest.raises(ValueError, match=field):
        ObjectBank({1: _net(), 5: _net(**kw)})


def test_num_graph_module_mismatch_raises():
    from checkerpose_b200.model.object_bank import ObjectBank
    other = _net()
    del other.refine_net[1].pre_query_block[2]
    with pytest.raises(ValueError, match="num_graph_module"):
        ObjectBank({1: _net(), 2: other})


def test_unknown_ids_raise_on_the_host():
    from checkerpose_b200.model.object_bank import ObjectBank
    bank = ObjectBank({1: _net(obj=1), 5: _net(obj=5)})
    feats = syn.synthetic_features(3, torch.Generator().manual_seed(0))
    with pytest.raises(ValueError, match=r"\[2\]"):
        bank(feats, torch.tensor([1, 2, 5]))
    g, order, groups = bank._order(torch.tensor([5, 1, 5, 1]), 4)
    assert g.tolist() == [1, 0, 1, 0] and order.tolist() == [1, 3, 0, 2] and groups == [(0, 0, 2), (1, 2, 4)]


def test_training_mode_raises():
    from checkerpose_b200.model.object_bank import ObjectBank
    bank = ObjectBank({1: _net()}).train()
    with pytest.raises(RuntimeError, match="inference-only"):
        bank(syn.synthetic_features(1, torch.Generator().manual_seed(0)), torch.tensor([1]))


_LAYOUT_C = r"""
#include <stddef.h>
#include <stdio.h>
#include "checkerpose_b200.h"
#define F(T, m) printf("%s.%s %zu\n", #T, #m, offsetof(T, m))
int main(void) {
  printf("cp_chain_layer %zu\n", sizeof(cp_chain_layer));
  F(cp_chain_layer, w_packed); F(cp_chain_layer, bias); F(cp_chain_layer, kin); F(cp_chain_layer, nout);
  F(cp_chain_layer, act); F(cp_chain_layer, slope); F(cp_chain_layer, w_stride); F(cp_chain_layer, b_stride);
  printf("cp_chain_params %zu\n", sizeof(cp_chain_params));
  F(cp_chain_params, layers); F(cp_chain_params, out_mode); F(cp_chain_params, out); F(cp_chain_params, n_valid);
  printf("cp_edgeconv_params %zu\n", sizeof(cp_edgeconv_params));
  F(cp_edgeconv_params, layer); F(cp_edgeconv_params, out_mode); F(cp_edgeconv_params, out); F(cp_edgeconv_params, n_valid);
  printf("cp_query_decode_params %zu\n", sizeof(cp_query_decode_params));
  F(cp_query_decode_params, perm); F(cp_query_decode_params, graph_sel); F(cp_query_decode_params, w1_stride);
  F(cp_query_decode_params, b1_stride); F(cp_query_decode_params, w2_stride); F(cp_query_decode_params, b2_stride);
  return 0;
}
"""


@pytest.mark.skipif(shutil.which("cc") is None, reason="no host C compiler")
def test_ctypes_layouts_match_the_header(tmp_path):
    import importlib.util
    spec = importlib.util.spec_from_file_location("_lib_structs", os.path.join(REPO, "checkerpose_b200", "_lib.py"))
    src = open(spec.origin).read().split("# name -> (restype, argtypes)")[0]      # the struct mirrors, without loading the .so
    ns = {"__name__": "_lib_structs"}
    exec(compile(src.replace("from .build import LIB_PATH", ""), spec.origin, "exec"), ns)
    (tmp_path / "layout.c").write_text(_LAYOUT_C)
    exe = tmp_path / "layout"
    subprocess.run(["cc", "-I", os.path.join(REPO, "include"), "-o", str(exe), str(tmp_path / "layout.c")], check=True)
    got = dict(line.rsplit(" ", 1) for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n") if line)
    py = {"cp_chain_layer": ns["ChainLayer"], "cp_chain_params": ns["ChainParams"], "cp_edgeconv_params": ns["EdgeConvParams"],
          "cp_query_decode_params": ns["QueryDecodeParams"]}
    for key, val in got.items():
        if "." in key:
            struct, member = key.split(".")
            assert getattr(py[struct], member).offset == int(val), key
        else:
            assert C.sizeof(py[key]) == int(val), key
