"""CPU-side tests: the C-ABI library loads and exports every symbol the header declares, the host
logic (state_dict layout, sharding, gather over gloo with world_size 2) works, and the product path
refuses CPU tensors instead of falling back."""
import ast
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import REPO, syn

torch.set_grad_enabled(False)


def header_functions():
    src = open(os.path.join(REPO, "include", "checkerpose_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(cp_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from checkerpose_b200 import _lib
    names = header_functions()
    assert len(names) >= 20
    for n in names:
        assert hasattr(_lib.lib, n), f"{n} declared in include/checkerpose_b200.h but not exported"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature"
    assert sorted(_lib.SIGNATURES) == names
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (cp_[a-z0-9_]+)", out))
    assert set(names) <= exported


# ctypes structure of checkerpose_b200/_lib.py -> its typedef in include/checkerpose_b200.h
ABI_STRUCTS = {
    "ChainLayer": "cp_chain_layer", "ChainParams": "cp_chain_params", "GraphPlanStruct": "cp_graph_plan",
    "EdgeConvParams": "cp_edgeconv_params", "GemmX3Params": "cp_gemm_x3_params", "ConvBf16Params": "cp_conv_bf16_params",
    "SlabPhase": "cp_slab_phase", "ConvSlabParams": "cp_conv_slab_params", "QueryDecodeParams": "cp_query_decode_params",
}


def test_ctypes_structures_match_the_header_layout(tmp_path):
    """Every parameter struct passed by pointer has the same size and field offsets in ctypes as in the C header (compiled
    with the host C compiler); a mismatch would otherwise only show on the GPU as garbage in the fields behind it."""
    import ctypes
    from checkerpose_b200 import _lib
    structs = sorted(n for n, v in vars(_lib).items() if isinstance(v, type) and issubclass(v, ctypes.Structure) and v is not ctypes.Structure)
    assert structs == sorted(ABI_STRUCTS)
    lines, expect = [], []
    for py_name, c_name in ABI_STRUCTS.items():
        cls = getattr(_lib, py_name)
        lines.append(f'printf("%zu\\n", sizeof({c_name}));')
        expect.append((c_name, ctypes.sizeof(cls)))
        for field, _ in cls._fields_:
            lines.append(f'printf("%zu %zu\\n", offsetof({c_name}, {field}), sizeof((({c_name}*)0)->{field}));')
            desc = getattr(cls, field)
            expect.append((f"{c_name}.{field} (offset, size)", f"{desc.offset} {desc.size}"))
    src = tmp_path / "layout.c"
    src.write_text("#include <stddef.h>\n#include <stdio.h>\n#include \"checkerpose_b200.h\"\nint main(void) {\n  "
                   + "\n  ".join(lines) + "\n  return 0;\n}\n")
    exe = tmp_path / "layout"
    cc = subprocess.run([os.environ.get("CC", "gcc"), "-std=c99", "-Wall", "-Werror", "-I", os.path.join(REPO, "include"),
                         "-o", str(exe), str(src)], capture_output=True, text=True)
    assert cc.returncode == 0, cc.stderr      # a ctypes field the header does not have fails here
    got = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines()
    assert len(got) == len(expect)
    for (what, want), line in zip(expect, got):
        assert line == str(want), f"{what}: header {line}, ctypes {want}"


def test_library_is_sm100a_with_blackwell_instructions():
    from checkerpose_b200 import _lib
    r = subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    assert "sm_100a" in r.stdout
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    for mnemonic in ("UTCHMMA", "UBLKCP", "LDTM"):  # tcgen05.mma, cp.async.bulk, tcgen05.ld
        assert mnemonic in sass, mnemonic


def test_error_reporting_without_gpu():
    from checkerpose_b200 import _lib
    assert _lib.lib.cp_version() >= 100
    assert _lib.lib.cp_packed_weight_bytes(256, 256) == 256 * 256 * 2
    assert _lib.lib.cp_packed_weight_bytes(7, 64) == 16 * 64 * 2      # rows padded to 16
    assert _lib.lib.cp_packed_weight_bytes(7, 60) == 0                # K must be a multiple of 64
    rc = _lib.lib.cp_knn(None, 1, 3, 10, 4, None, None, None)
    assert rc == -1 and b"null" in _lib.lib.cp_last_error_string()
    with pytest.raises(RuntimeError):
        _lib.check(rc, "cp_knn")


def test_no_cpu_fallback():
    from checkerpose_b200 import ops
    from checkerpose_b200.model import pipeline
    x = torch.randn(1, 3, 32)
    for fn in (lambda: ops.knn(x, 4), lambda: pipeline.knn(x, 4), lambda: pipeline.from_mask_prob_to_mask(x),
               lambda: pipeline.from_code_prob_to_id(x), lambda: ops.threshold(x)):
        with pytest.raises(RuntimeError, match="CUDA"):
            fn()


def test_product_never_imports_the_oracle():
    pkg = os.path.join(REPO, "checkerpose_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if not f.endswith(".py"):
                continue
            tree = ast.parse(open(os.path.join(root, f)).read())
            for node in ast.walk(tree):
                mods = []
                if isinstance(node, ast.Import):
                    mods = [a.name for a in node.names]
                elif isinstance(node, ast.ImportFrom):
                    mods = [node.module or ""]
                assert not any(m.split(".")[0] == "oracle" for m in mods), f"{f} imports oracle/"


def test_state_dict_layout_matches_reference_keys():
    """Keys/shapes == the layout the reference modules loaded strictly in tests/golden/make_golden.py."""
    from checkerpose_b200.model import init, init_lm, pipeline, pipeline_lm
    from checkerpose_b200.model.backbone import FeatureListBackbone
    N = 64
    p3d = syn.p3d_normed_tensor(syn.load_fps_xyz("lmo", 1, N))
    for I, P in ((init, pipeline), (init_lm, pipeline_lm)):
        inet = I.InitNet_GNN(npoint=N, p3d_normed=p3d, res_log2=3, backbone_name="hrnet_w18", pretrain_backbone=False,
                             img_backbone=FeatureListBackbone())
        net = P.PoseNet_GNNskip(inet, npoint=N, p3d_normed=p3d, res_log2=6, local_k=2, num_graph_module=3)
        want = {k: tuple(s) for k, s, _, _ in syn.head_param_spec(N)}
        got = {k: tuple(v.shape) for k, v in net.state_dict().items()}
        assert want == got
        assert "knn_idx" not in "".join(got)            # plain attribute, not a buffer (reference: pipeline.py:48)
        net.load_state_dict(syn.synthetic_state_dict(syn.head_param_spec(N), torch.Generator().manual_seed(0)), strict=True)
        net.eval()
        with pytest.raises(RuntimeError):                # built on CPU: the graph needs a GPU, no CPU kNN
            feats = syn.synthetic_features(1, torch.Generator().manual_seed(0))
            net(feats, p3d, torch.tensor([1])) if P is pipeline_lm else net(feats, p3d)
    bare = init.InitNet_GNN(npoint=N, p3d_normed=p3d, backbone_name="hrnet_w18", img_backbone=FeatureListBackbone())
    want = {k: tuple(s) for k, s, _, _ in syn.head_param_spec(N, include_refine=False, prefix_init="")}
    assert want == {k: tuple(v.shape) for k, v in bare.state_dict().items()}


def test_abwoprog_state_dict_layout_and_reference_import_surface():
    """pipeline_lm exports what test_lm.py:27 / train_lm.py:23 import, and the ablation net's state_dict layout is the one
    the unmodified reference module loaded in tests/golden/make_golden.py::golden_abwoprog."""
    from checkerpose_b200.model import init_lm, pipeline_lm
    from checkerpose_b200.model.backbone import FeatureListBackbone
    from checkerpose_b200.model.pipeline_lm import PoseNet_GNNskip, PoseNet_GNNskip_ABwoProg  # noqa: F401  (the reference's import line)
    N = 64
    p3d = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz("lm", o, N)) for o in (1, 2)], dim=0)
    inet = init_lm.InitNet_GNN(npoint=N, p3d_normed=p3d, res_log2=3, backbone_name="hrnet_w18", pretrain_backbone=False,
                               img_backbone=FeatureListBackbone())
    net = pipeline_lm.PoseNet_GNNskip_ABwoProg(inet, npoint=N, p3d_normed=p3d, res_log2=6, local_k=2, num_graph_module=3)
    want = {k: tuple(s) for k, s, _, _ in syn.abwoprog_param_spec(N)}
    got = {k: tuple(v.shape) for k, v in net.state_dict().items()}
    assert want == got
    assert got["query_block.mlps.4.weight"] == (13, 64)      # one query for all 2 * res_log2 + 1 bits


def test_fps_dropin_needs_gpu():
    from checkerpose_b200.preprocess_data.get_fps_points import farthest_point_sample_init_center
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    with pytest.raises(RuntimeError):
        farthest_point_sample_init_center(np.zeros((10, 3)), 4)


def test_synthetic_generators_are_deterministic():
    a = syn.synthetic_state_dict(syn.head_param_spec(64), torch.Generator().manual_seed(5))
    b = syn.synthetic_state_dict(syn.head_param_spec(64), torch.Generator().manual_seed(5))
    assert all(torch.equal(a[k], b[k]) for k in a)
    gam = a["refine_net.0.pre_query_block.0.conv.1.weight"]
    assert (gam < 0).any() and (gam > 0).any(), "negative BN gammas must be exercised"
    xyz = syn.load_fps_xyz("ycbv", 21, 4096)
    assert xyz.shape == (4096, 3) and np.array_equal(syn.load_fps_xyz("ycbv", 21, 512), xyz[:512])
    pn = syn.pc_normalize(xyz.copy())
    assert abs(np.sqrt((pn ** 2).sum(1)).max() - 1.0) < 1e-12 and np.abs(pn.mean(0)).max() < 1e-12


def test_shard_ranges():
    from checkerpose_b200.dist import shard_range, shard_sizes
    for total in (0, 1, 7, 256, 1024, 1000):
        for world in (1, 2, 3, 4, 8):
            spans = [shard_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = shard_sizes(total, world)
            assert max(sizes) - min(sizes) <= 1 and sum(sizes) == total


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, {repo!r})
from checkerpose_b200.dist import gather_correspondences, shard_range
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=rank, world_size=world)
for total in (8, 7):
    N = 5
    full = torch.arange(total * N * 3, dtype=torch.int32).view(total, N, 3)
    lo, hi = shard_range(total, rank, world)
    got = gather_correspondences(full[lo:hi].clone(), total=total)
    assert got.shape == full.shape and torch.equal(got, full), (rank, total)
dist.barrier()
dist.destroy_process_group()
print("ok", rank)
"""


def test_gather_correspondences_gloo_world2(tmp_path):
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(repo=REPO, port=port))
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    for p in procs:
        out, _ = p.communicate(timeout=120)
        assert p.returncode == 0 and "ok" in out, out


def test_bench_reference_arm_contract():
    """--impl reference must print one JSON line with the agreed keys (tiny steps to stay fast is not possible:
    one N=4096 RoI takes seconds on CPU, so only the argument plumbing is checked here)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench", os.path.join(REPO, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    assert bench.METRIC.startswith("RoIs/sec") and "4096" in bench.METRIC
    hbm, tf_burst, tf_sus, src = bench.load_peaks()
    assert hbm > 1000 and tf_burst >= tf_sus > 100 and ("measured" in src or "fallback" in src)
    # every BASELINE config is a workload of the bench; the default is configs[2]
    import argparse
    for name, per_gpu, scaling in (("full4096", 256, "weak"), ("init64", 64, "weak"), ("ycbv1024", 128, "strong"), ("lm_sweep", 256, "weak")):
        wl = bench.workload(argparse.Namespace(config=name, npoint=0, graph_k=0, batch=0), world=8)
        assert wl["per_gpu"] == per_gpu and wl["scaling"] == scaling
    assert bench.LM_OBJECT_IDS == (1, 2, 4, 5, 6, 8, 9, 10, 11, 12, 13, 14, 15)


def test_bench_dump_outputs_float32_and_seeded_sample(tmp_path, monkeypatch):
    """--dump-outputs: one float32 .npy per tensor the step returned (packed records unpacked); above the byte budget,
    the same fixed seeded sample of RoIs from every array, listed in roi_rows.npy."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench", os.path.join(REPO, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    B, N = 16, 64
    g = torch.Generator().manual_seed(0)
    last = dict(roi_bit=torch.randn(B, 1, N, generator=g), x_bits=torch.randn(B, 6, N, generator=g),
                y_bits=torch.randn(B, 6, N, generator=g), seg=torch.randn(B, 2, 64, 64, generator=g),
                x_id=torch.randint(0, 64, (B, N), generator=g), y_id=torch.randint(0, 64, (B, N), generator=g),
                records=torch.zeros(B, 16 + 2 * N, dtype=torch.uint8))

    def dump(name):
        bench.dump_outputs(str(tmp_path / name), last)
        return {f[:-4]: np.load(tmp_path / name / f) for f in os.listdir(tmp_path / name)}
    full = dump("full")
    assert sorted(full) == ["records_flags", "records_uv", "roi_bit", "roi_rows", "seg", "x_bits", "x_id", "y_bits", "y_id"]
    assert all(a.dtype == np.float32 and len(a) == B for k, a in full.items() if k != "roi_rows")
    assert np.array_equal(full["roi_rows"], np.arange(B)) and full["records_uv"].shape == (B, N, 2)
    assert np.array_equal(full["x_bits"], last["x_bits"].numpy()) and np.array_equal(full["y_id"], last["y_id"].numpy())
    per_roi = sum(a[0].nbytes for a in full.values())
    monkeypatch.setattr(bench, "DUMP_BUDGET_BYTES", 5 * per_roi)
    a, b = dump("a"), dump("b")
    rows = a["roi_rows"].astype(np.int64)
    assert len(rows) == 5 and np.array_equal(np.unique(rows), rows) and sum(x.nbytes for x in a.values()) <= 5 * per_roi
    for k in full:
        assert np.array_equal(a[k], b[k]) and (k == "roi_rows" or np.array_equal(a[k], full[k][rows])), k


# ------------------------------------------------------------------------------------------------ graph plan (host code)
@pytest.mark.parametrize("ds,objs,N,K", [("lmo", (1,), 4096, 20), ("ycbv", (21,), 512, 20), ("lm", (2, 9), 300, 8), ("lmo", (5,), 1024, 40),
                                         ("lmo", (8,), 200, 13)])
def test_graph_plan_invariants(ds, objs, N, K):
    """cp_graph_plan_build: the renumbering is a permutation, the plan-order neighbour table, the per-tile staging lists
    and the node-pair programs reproduce the reference graph exactly, and FPS clouds fit the staged kernel's ring."""
    from checkerpose_b200 import ops
    from checkerpose_b200 import synthetic as syn
    from oracle import checkerpose_oracle as orc
    p3d = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz(ds, o, N)) for o in objs], dim=0)
    idx = orc.knn(p3d, K)                                   # (G,N,K) int64, keypoint numbering
    plan = ops.GraphPlan(idx.to(torch.int32), p3d)
    G, KP, TILE = len(objs), plan.KP, ops.PLAN_TILE
    assert KP >= K and KP % 4 == 0 and plan.PW == 2 * KP + 8
    assert plan.staged == (plan.max_unique <= min(ops.PLAN_UMAX, plan.ring_rows)) and (plan.staged or K > 20), plan.max_unique
    perm = plan.perm.long()
    saved = total = 0
    for g in range(G):
        assert torch.equal(torch.sort(perm[g])[0], torch.arange(N))
        # same edges: keypoint ids of the plan-order neighbours == the reference's neighbours of that keypoint
        assert torch.equal(perm[g][plan.idx_p[g].long()], idx[g][perm[g]])
        for t in range(plan.T):
            n0, n1 = t * TILE, min(N, (t + 1) * TILE)
            U = int(plan.ucount[g, t])
            want_u = torch.unique(plan.idx_p[g, n0:n1].long())
            assert U == len(want_u)
            if U > ops.PLAN_UMAX:
                continue   # list truncated: the caller must not use the staged kernel (plan.staged is False)
            ul = (plan.ulist[g, t].long() & 0xFFFF).t().reshape(-1)      # entry [q][i] is list position 64 i + q
            assert torch.equal(ul[:U], want_u) and bool((ul[U:] == 0xFFFF).all())
            prog = plan.prog[g, t].long() & 0xFFFF            # (64, PW)
            assert bool((prog[:, :2 * KP] % 128 == 0).all())
            rows = ul[(prog[:, :2 * KP] // 128).clamp(max=U - 1)]   # staged row of every program entry
            a_id, b_id, C = prog[:, 2 * KP] & 255, prog[:, 2 * KP] >> 8, prog[:, 2 * KP + 1]
            assert bool((C % 4 == 0).all()) and bool((C.view(-1, 4) == C.view(-1, 4)[:, :1]).all())   # uniform per warp
            seen = []
            for q in range(ops.PLAN_PAIRS):
                c = int(C[q])
                if int(a_id[q]) == 255:
                    assert int(b_id[q]) == 255
                    continue
                na = set(plan.idx_p[g, n0 + int(a_id[q])].tolist())
                assert set(rows[q, :KP].tolist()) == na              # a-list (with padding) == a's neighbour set
                seen.append(int(a_id[q]))
                total += 2 * KP
                if int(b_id[q]) != 255:
                    nb = set(plan.idx_p[g, n0 + int(b_id[q])].tolist())
                    common = set(rows[q, :c].tolist())
                    assert len(common) == c and common <= nb         # the first C rows of a are shared with b
                    assert common | set(rows[q, KP:2 * KP - c].tolist()) == nb
                    seen.append(int(b_id[q]))
                    saved += c
            assert sorted(seen) == list(range(n1 - n0))               # every node of the tile exactly once
    # locality is the point of the renumbering: far fewer distinct rows per tile than K * 128 ...
    assert plan.max_unique < 0.3 * TILE * K or N <= 512
    # ... and neighbouring nodes share neighbours: the pair programs skip a good part of the row reads
    if N >= 1024 and K >= 20:
        assert saved / total > 0.25, saved / total


def test_graph_plan_without_coordinates_keeps_order():
    from checkerpose_b200 import ops
    g = torch.Generator().manual_seed(0)
    idx = torch.randint(0, 2000, (1, 2000, 12), generator=g, dtype=torch.int32)
    plan = ops.GraphPlan(idx, None)
    assert plan.identity and torch.equal(plan.idx_p, idx) and not plan.staged   # random graph: too many distinct rows


def test_cache_keys_tolerate_inference_tensors():
    """ADVICE r1: tensors created under torch.inference_mode() raise when ``_version`` is read; the prepared-weight and
    graph caches must not."""
    from checkerpose_b200 import head
    with torch.inference_mode():
        lin = torch.nn.Linear(8, 4)
        t = torch.arange(6).view(1, 2, 3)
    assert t.is_inference()
    with pytest.raises(RuntimeError):
        t._version
    assert head._ver(t) == -1 and head._ver(torch.zeros(2)) == 0
    fp = head._param_fingerprint(lin)
    assert len(fp) == 2 and fp == head._param_fingerprint(lin)


def test_rgb_image_to_class_id_image():
    from checkerpose_b200.binary_code_helper import class_id_encoder_decoder as codec
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, size=(5, 7, 3), dtype=np.uint8)
    ids = codec.RGB_image_to_class_id_image(img)
    want = img[..., 0].astype(np.int64) * 65536 + img[..., 1].astype(np.int64) * 256 + img[..., 2].astype(np.int64)
    assert ids.shape == (5, 7) and np.array_equal(ids, want)


def test_product_package_does_not_read_tests_dir():
    pkg = os.path.join(REPO, "checkerpose_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py") and "make_fps_fixture" not in f:
                src = open(os.path.join(root, f)).read()
                assert '"tests"' not in src and "'tests'" not in src, f"{f} refers to the tests directory"
    assert os.path.exists(syn.FPS_FIXTURE) and os.sep + "tests" + os.sep not in syn.FPS_FIXTURE


def test_negative_leaky_slope_is_rejected_by_the_fold():
    """lrelu(max_k P + Q) == max_k lrelu(P + Q) needs an increasing activation (ADVICE r1)."""
    from checkerpose_b200 import head
    src = open(os.path.join(REPO, "checkerpose_b200", "head.py")).read()
    assert "negative_slope >= 0" in src and hasattr(head, "PreparedEdgeConv")
