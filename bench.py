#!/usr/bin/env python
"""Benchmark of the GNN keypoint head (BASELINE.json metric: RoIs/sec, 4096-keypoint head).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dtype bf16|fp32]
                  [--config full4096|init64|ycbv1024|lm_sweep] [--dump-outputs DIR]

One "step" = one pass of the post-backbone head over a batch of synthetic RoIs.  Default workload (the headline):
BASELINE.json configs[2], "full progressive 512->4096 keypoint GNN head, batch 256 RoIs, bf16" -- 256 RoIs PER GPU
(weak scaling: the RoI batch is sharded, weights and graph replicated); with N > 1 one NCCL all-gather of the decoded
correspondence records per step, issued on a side stream and overlapped with the next step (completed inside the timed
region).  The other BASELINE configs are behind --config (their lines are committed under profiles/):

  init64    configs[1]: init_gnn2_hrnetw18_npt512 head (512 keypoints, 7 low-level bits), 64 RoIs, 1 GPU
  ycbv1024  configs[3]: 21 YCB-V objects = 21 graphs selected per RoI (pipeline_lm API), 1024 RoIs in total
            sharded over the GPUs (STRONG scaling), records gathered over NVLink
  lm_sweep  configs[4]: LM single-model net (15 graphs, ids from the 13-object list), keypoint-count x graph_k sweep

Prints ONE JSON line (rank 0).  ``value`` = RoIs/s with inputs resident in HBM; ``e2e`` = the same through the public
module API from pinned host buffers (H2D of the feature maps the head reads + D2H of the records every step);
``roofline`` = the dominant kernel (fused EdgeConv aggregation + [P|Q] GEMM, edgeconv_kernel) timed live with CUDA
events on its launching stream; ``roofline_k3`` = the sampling + pre-graph MLP kernel; ``gnn_only`` = the step without
the library convolutions of the image branch; ``parity`` = agreement of the decoded correspondences with the CPU oracle
on a small sample, computed outside every timed region; ``cpu_baseline`` = the CPU restatement of the reference head on
this box's host cores over a bounded sample.  ``--impl reference`` times only the CPU arm (the unmodified reference
modules when /root/reference is present, else the oracle port; the line says which).

``--dump-outputs DIR`` writes, after the timed steps, what the last timed step returned to its caller as float32 .npy files
(a fixed seeded sample of the RoIs when the batch is larger than 60 MiB).  Inputs and weights come from fixed seeds, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import torch  # noqa: E402

METRIC = "RoIs/sec (4096-kpt GNN head)"
UNIT = "RoIs/s"
GRAPH_K = 20
# dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel, from the committed
# `ncu --set full` capture of this command (profiles/)
DOMINANT_KERNEL_DRAM_BYTES = 1.077e9 + 1.022e9
DOMINANT_KERNEL_DRAM_SOURCE = "profiles/r02_h_edgeconv.txt (ncu --set full of bench.py --profile, launch 0: dram read 1.077 GB + write 1.022 GB)"
K3_KERNEL_DRAM_BYTES = 0.567e9 + 1.022e9
K3_KERNEL_DRAM_SOURCE = "profiles/r02_h_taps_chain_query_tail.txt (ncu --set full, launch 0: dram read 0.567 GB + write 1.022 GB)"
LM_OBJECT_IDS = (1, 2, 4, 5, 6, 8, 9, 10, 11, 12, 13, 14, 15)     # the 13 LM objects of test_lm.py:109
DUMP_BUDGET_BYTES = 60 << 20      # --dump-outputs writes at most this much (plus the .npy headers): under 64 MB


def load_peaks():
    """-> (hbm GB/s, bf16 TFLOP/s burst, bf16 TFLOP/s sustained, source)."""
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d["bf16_tflops"]), float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), \
            "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1590.0, 1400.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                smax.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------------
def workload(args, world):
    """-> dict describing the --config: dataset / objects / N / K / RoIs per GPU / scaling / which nets."""
    c = args.config
    if c == "full4096":
        return dict(name=c, ds="lmo", objs=(1,), lm=False, N=args.npoint or 4096, K=args.graph_k or GRAPH_K,
                    per_gpu=args.batch or 256, scaling="weak", init_only=False,
                    text="full progressive head (init net + 3 refine stages + decode + correspondences), N=4096 keypoints, "
                         "K=20, 256 RoIs per GPU (BASELINE.json configs[2])")
    if c == "init64":
        return dict(name=c, ds="lmo", objs=(1,), lm=False, N=args.npoint or 512, K=args.graph_k or GRAPH_K,
                    per_gpu=args.batch or 64, scaling="weak", init_only=True,
                    text="init_gnn2_hrnetw18_npt512 head: conv1x1 + 2 EdgeConv(64) + Linear(64->7) + decode of the 7 low-level bits, "
                         "N=512 keypoints, 64 RoIs (BASELINE.json configs[1])")
    if c == "ycbv1024":
        total = args.batch or 1024
        assert total % world == 0, "ycbv1024: the RoI count must divide by the number of GPUs"
        return dict(name=c, ds="ycbv", objs=tuple(range(1, 22)), lm=True, N=args.npoint or 4096, K=args.graph_k or GRAPH_K,
                    per_gpu=total // world, scaling="strong", init_only=False,
                    text=f"YCB-V converted config: 21 objects = 21 kNN graphs selected per RoI (pipeline_lm API), {total} RoIs in total "
                         f"sharded over the GPUs, records gathered over NVLink (BASELINE.json configs[3])")
    if c == "lm_sweep":
        return dict(name=c, ds="lm", objs=tuple(range(1, 16)), lm=True, N=args.npoint or 4096, K=args.graph_k or GRAPH_K,
                    per_gpu=args.batch or 256, scaling="weak", init_only=False,
                    text="LM single-model net: 15 graphs, per-RoI object ids from the 13-object list (test_lm.py:109), "
                         "keypoint-count x graph_k sweep (BASELINE.json configs[4])")
    raise ValueError(c)


def build_case(wl, dev, seed_rank, N=None, K=None, batch=None):
    """Nets, weights and the synthetic RoI batch of a workload on ``dev``."""
    from checkerpose_b200 import synthetic as syn
    from checkerpose_b200.model import init, init_lm, pipeline, pipeline_lm
    from checkerpose_b200.model.backbone import FeatureListBackbone
    N, K, B = N or wl["N"], K or wl["K"], batch or wl["per_gpu"]
    g = torch.Generator().manual_seed(1234 + 2)
    p3d = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz(wl["ds"], o, N)) for o in wl["objs"]], dim=0).to(dev)
    I, P = (init_lm, pipeline_lm) if wl["lm"] else (init, pipeline)
    if wl["init_only"]:
        sd = syn.synthetic_state_dict(syn.head_param_spec(N, include_refine=False, prefix_init=""), g)
        net = I.InitNet_GNN(npoint=N, p3d_normed=p3d, res_log2=3, backbone_name="hrnet_w18", pretrain_backbone=False,
                            max_batch_size=B, num_graph_module=2, graph_k=K, img_backbone=FeatureListBackbone())
    else:
        sd = syn.synthetic_state_dict(syn.head_param_spec(N), g)
        inet = I.InitNet_GNN(npoint=N, p3d_normed=p3d, res_log2=3, backbone_name="hrnet_w18", pretrain_backbone=False,
                             max_batch_size=B, num_graph_module=2, graph_k=K, img_backbone=FeatureListBackbone())
        net = P.PoseNet_GNNskip(inet, npoint=N, p3d_normed=p3d, res_log2=6, num_filters=256, max_batch_size=B,
                                local_k=2, leaky_slope=0.01, num_graph_module=3, graph_k=K)
    net.load_state_dict(sd, strict=True)
    net = net.to(dev).eval()
    obj_ids = None
    if wl["lm"]:
        pool = LM_OBJECT_IDS if wl["ds"] == "lm" else wl["objs"]
        go = torch.Generator().manual_seed(777 + seed_rank)
        obj_ids = torch.tensor(pool)[torch.randint(0, len(pool), (B,), generator=go)].to(dev)
    return dict(net=net, sd=sd, p3d=p3d, obj_ids=obj_ids, N=N, K=K, B=B, init_only=wl["init_only"])


def make_inputs(case, dev, dtype, seed_rank):
    """Synthetic RoI batch, distinct per rank and per RoI.  The head reads img_feats[-1], [-2], [-3] only
    (pipeline.py:361,372 -- the 128 x 64 x 64 HRNet map is never touched), so only those three are created / uploaded."""
    from checkerpose_b200 import synthetic as syn
    B = case["B"]
    gg = torch.Generator(device=dev).manual_seed(4321 + seed_rank)
    first = 3 if case.get("init_only") else 1      # the init net alone reads only the 1024 x 8 x 8 map (init.py:111-112)
    feats = [torch.relu(torch.randn(B, c, s, s, generator=gg, device=dev)).to(dtype)
             for c, s in zip(syn.HRNET_W18_DIMS[first:], syn.HRNET_W18_SIZES[first:])]
    bbox = syn.synthetic_bboxes(B, torch.Generator().manual_seed(99 + seed_rank)).to(dev)
    return feats, bbox


def make_step(wl, case, bbox, gather, last=None):
    """-> step(feats) -> (records or logits, done_event).  The records leave in the packed 2-byte form.  With a dict
    ``last``, every step leaves there the tensors its caller receives (for --dump-outputs)."""
    net, obj_ids = case["net"], case["obj_ids"]
    pexp = case["p3d"][obj_ids - 1] if wl["lm"] else case["p3d"].expand(case["B"], -1, -1)
    if wl["init_only"]:
        from checkerpose_b200.model import pipeline as P

        def step(f):
            bits = net(f, obj_ids) if wl["lm"] else net(f)
            # decode of the low-level bits (pipeline.py:363-369): roi mask + 3+3-bit cell ids
            mask = P.from_mask_prob_to_mask(bits[:, 0:1].contiguous())
            x_id = P.from_code_prob_to_id(bits[:, 1:4].contiguous())
            ids = P.from_code_prob_to_id(bits[:, 4:7].contiguous())
            if last is not None:
                last.update(init_bits=bits, roi_mask=mask, x_id=x_id, y_id=ids)
            ev = torch.cuda.Event()
            ev.record()
            return ids, ev
        return step

    def step(f):
        out, corr = net.forward_with_correspondences(f, pexp, bbox, obj_ids=obj_ids, packed=True)
        if last is not None:
            last.update(zip(("roi_bit", "x_bits", "y_bits", "seg", "x_id", "y_id"), out), records=corr)
        return gather.submit(corr)
    return step


def dump_outputs(out_dir, last):
    """--dump-outputs: write the tensors of ``last`` as ``out_dir/<name>.npy`` in float32.  The packed correspondence records
    are unpacked into what their consumer reads (records_uv, records_flags).  If the whole batch exceeds DUMP_BUDGET_BYTES,
    a fixed seeded sample of RoIs is written instead: the same rows of every array, listed in roi_rows.npy."""
    import numpy as np
    from checkerpose_b200 import ops
    host = {}
    for name, t in last.items():
        if name == "records":
            uv, flags, _, _, _ = ops.unpack_correspondences_host(t)
            host["records_uv"], host["records_flags"] = uv, flags.astype(np.float32)
        else:
            host[name] = t.float().cpu().numpy()
    B = len(host["x_id"])
    per_roi = sum(a[0].nbytes for a in host.values()) + 8          # + its entry in roi_rows.npy
    rows = np.arange(B)
    if B * per_roi > DUMP_BUDGET_BYTES:
        rows = np.sort(torch.randperm(B, generator=torch.Generator().manual_seed(0))[:DUMP_BUDGET_BYTES // per_roi].numpy())
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a[rows]))
    np.save(os.path.join(out_dir, "roi_rows.npy"), rows.astype(np.float64))


# ------------------------------------------------------------------------------------------------------
# CPU arm: the unmodified reference when it is present (build container), else the oracle port
# ------------------------------------------------------------------------------------------------------
def cpu_reference_rois_per_s(steps, warmup, N=4096, K=GRAPH_K, rois_per_step=1, budget_s=None):
    """-> (RoIs/s, timed steps, ms per step, kind).  Same synthetic weights / keypoints / feature shapes as the GPU arm."""
    from checkerpose_b200 import synthetic as syn
    torch.set_grad_enabled(False)
    torch.set_num_threads(os.cpu_count() or 1)
    g = torch.Generator().manual_seed(1234 + 2)
    p3d = syn.p3d_normed_tensor(syn.load_fps_xyz("lmo", 1, N))
    sd = syn.synthetic_state_dict(syn.head_param_spec(N), g)
    feats = syn.synthetic_features(rois_per_step, g)
    kind = "port"
    if os.path.isdir("/root/reference/checkerpose/model"):
        try:
            from oracle import reference_runner
            run = reference_runner.build_reference_head(N, K, p3d, sd, rois_per_step)
            kind = "reference"
        except Exception as e:        # a broken stub must not take the bench down: fall back to the port and say so
            print(f"bench.py: unmodified reference unavailable ({type(e).__name__}: {e}); timing the oracle port", file=sys.stderr)
    if kind == "port":
        from oracle import checkerpose_oracle as orc
        idx = orc.knn(p3d, K)

        def run(f):
            return orc.pose_head(f, sd, idx, [idx] * 3, N)
    times = []
    t_start = time.perf_counter()
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        run(feats)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
        if budget_s is not None and times and time.perf_counter() - t_start > budget_s:
            break
    total = sum(times)
    return rois_per_step * len(times) / total, len(times), total / len(times) * 1e3, kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    v, n, ms, kind = cpu_reference_rois_per_s(args.steps, args.warmup, rois_per_step=1)
    what = "unmodified reference modules (/root/reference, timm stubbed)" if kind == "reference" else "CPU port of the reference (oracle/)"
    sample = f"{n} timed steps x 1 RoI (N=4096, K={GRAPH_K}) of the same workload, fp32, torch CPU ops, {cores} threads; {what}"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": n, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"full progressive head, N=4096 keypoints, K=20, 3 refine stages (BASELINE.json configs[2]); {what}, 1 RoI per step",
                   "same_config_as_gpu_arm": False,
                   "note": "the GPU arm runs 256 RoIs per step per GPU; the CPU arm materialises 168 MB per RoI per EdgeConv layer and runs 1 RoI per step"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------------
def parity_sample(wl, case, feats, bbox, dtype, nroi=2):
    """Decoded correspondences of the first ``nroi`` RoIs of this rank's batch against the CPU oracle on the same tensors
    (outside every timed region; the oracle is the checker, never the thing measured)."""
    from checkerpose_b200 import ops
    from oracle import checkerpose_oracle as orc
    net, N, K = case["net"], case["N"], case["K"]
    f2 = [f[:nroi].contiguous() for f in feats]
    obj = None if case["obj_ids"] is None else case["obj_ids"][:nroi]
    pexp = case["p3d"][obj - 1] if wl["lm"] else case["p3d"].expand(nroi, -1, -1)
    (roi, xb, yb, seg, xid, yid), packed = net.forward_with_correspondences(f2, pexp, bbox[:nroi].contiguous(), obj_ids=obj, packed=True)
    torch.cuda.synchronize()
    uv, flags, x2, y2, _ = ops.unpack_correspondences_host(packed)
    sd = {k: v.float() for k, v in case["sd"].items()}
    idx = orc.knn(case["p3d"].float().cpu(), K)
    cf = [torch.zeros(nroi, 128, 64, 64)] + [f.float().cpu() for f in f2]
    ref = orc.pose_head(cf, sd, idx, [idx] * 3, N, obj_ids=None if obj is None else obj.cpu())
    rx, ry = ref[4].numpy(), ref[5].numpy()
    cell = float(((x2 == rx) & (y2 == ry)).mean())
    stage = [float((((x2 >> (6 - L)) == (rx >> (6 - L))) & ((y2 >> (6 - L)) == (ry >> (6 - L)))).mean()) for L in (3, 4, 5, 6)]
    roi_ok = float((((flags & 1) != 0) == (ref[0][:, 0].numpy() > 0)).mean())
    return {"keypoint_agreement": cell, "agreement_after_stage": {"init(8x8)": stage[0], "refine0(16x16)": stage[1],
                                                                    "refine1(32x32)": stage[2], "refine2(64x64)": stage[3]},
            "roi_bit_agreement": roi_ok, "sample": f"{nroi} RoIs x {N} keypoints of this run's batch vs oracle.pose_head (fp32, CPU) on the same tensors",
            "note": ("bf16 mode: every tensor between layers is re-quantised to bf16 and 13 cascaded sign tests sit on random-init logits; "
                     "the >= 99.9 % bar is held by --dtype fp32 (DESIGN.md section 6)") if dtype == torch.bfloat16 else
                    "float32 mode (split-bf16 tensor-core GEMMs, fp32 storage)"}


def kernel_rooflines(log, ms_total, steps, B, N, dtype, world):
    """Live rooflines of the two big kernels from the per-launch CUDA events of the timed loop."""
    from checkerpose_b200 import ops
    hbm, tf_burst, tf_sus, peak_src = load_peaks()
    s_el = 2 if dtype == torch.bfloat16 else 4

    def is_dom(sig):
        return sig[0] in ("EC", ops.PRO_AGG) and sig[1] == 256 and sig[2] == (512,)
    dom = [a.elapsed_time(b) for sig, a, b in log if is_dom(sig)]
    allchain = sum(a.elapsed_time(b) for _, a, b in log)
    roof = None
    if dom:
        dom_name = "edgeconv_kernel" if any(sig[0] == "EC" for sig, _, _ in log if is_dom(sig)) else "chain_kernel<AGG>"
        avg_ms = sum(dom) / len(dom)
        alg_bytes = B * (N * 256 * s_el + N * 256 * s_el)          # SURVEY 8(d): N*C*s + N*C'*s per RoI-layer
        alg_flops = 2.0 * B * N * 256 * 512                         # factored formulation: one 256 -> [P|Q] 512 GEMM per node
        t_hbm, t_tensor = alg_bytes / (hbm * 1e9) * 1e3, alg_flops / (tf_sus * 1e12) * 1e3
        ach_b, ach_f = alg_bytes / (avg_ms * 1e-3) / 1e9, alg_flops / (avg_ms * 1e-3) / 1e12
        bound = "tensor" if t_tensor > t_hbm else "hbm"
        roof = {"bound": bound, "kernel": f"{dom_name} (EdgeConv max-aggregation + [P|Q] GEMM, C=256, factored formulation)",
                "achieved": ach_f if bound == "tensor" else ach_b, "peak": tf_sus if bound == "tensor" else hbm,
                "unit": "TFLOP/s" if bound == "tensor" else "GB/s", "frac": max(t_hbm, t_tensor) / avg_ms,
                "peak_source": peak_src + (", sustained bf16 (kernel timed inside a long step)" if bound == "tensor" else ""),
                "rule": "SURVEY 8(d): bound = argmax(flops / peak_tensor, bytes / peak_hbm); frac = that time / measured launch time",
                "hbm": {"achieved": ach_b, "peak": hbm, "unit": "GB/s", "frac": ach_b / hbm, "algorithmic_bytes_per_launch": alg_bytes},
                "tensor": {"achieved": ach_f, "peak": tf_sus, "unit": "TFLOP/s", "frac": ach_f / tf_sus, "algorithmic_flops_per_launch": alg_flops},
                "traffic": DOMINANT_KERNEL_DRAM_BYTES, "traffic_source": DOMINANT_KERNEL_DRAM_SOURCE,
                "avg_launch_ms": avg_ms, "launches_per_step": len(dom) / steps,
                "share_of_step": sum(dom) / ms_total if world == 1 else None,
                "all_gnn_kernels_share_of_step": allchain / ms_total if world == 1 else None}
    k3 = [a.elapsed_time(b) for sig, a, b in log if sig[0] == ops.PRO_TAPS and sig[1] == 512]
    roof_k3 = None
    if k3:
        k3_ms = sum(k3) / len(k3)
        # SURVEY 8(d): min((H+1)^2 * 64, 4 * 64 * N) patch elements + graph feature read, [P|Q] written; the two launches
        # timed here are refine stages 1 and 2 (H = 32, 64): per-launch average
        k3_bytes = B * s_el * (N * (256 + 512) + (min(33 * 33 * 64, 256 * N) + min(65 * 65 * 64, 256 * N)) // 2)
        k3_flops = 2.0 * B * N * (512 * 256 + 256 * 256 + 256 * 512)
        t_hbm, t_tensor = k3_bytes / (hbm * 1e9) * 1e3, k3_flops / (tf_sus * 1e12) * 1e3
        bound = "tensor" if t_tensor > t_hbm else "hbm"
        ach_b, ach_f = k3_bytes / (k3_ms * 1e-3) / 1e9, k3_flops / (k3_ms * 1e-3) / 1e12
        roof_k3 = {"bound": bound, "kernel": "taps_chain_kernel (4-tap gather x mask | graph feature -> MLP x2 -> [P|Q] GEMM)",
                   "achieved": ach_f if bound == "tensor" else ach_b, "peak": tf_sus if bound == "tensor" else hbm,
                   "unit": "TFLOP/s" if bound == "tensor" else "GB/s", "frac": max(t_hbm, t_tensor) / k3_ms, "peak_source": peak_src,
                   "hbm": {"achieved": ach_b, "peak": hbm, "frac": ach_b / hbm, "algorithmic_bytes_per_launch": k3_bytes},
                   "tensor": {"achieved": ach_f, "peak": tf_sus, "frac": ach_f / tf_sus, "algorithmic_flops_per_launch": k3_flops},
                   "traffic": K3_KERNEL_DRAM_BYTES, "traffic_source": K3_KERNEL_DRAM_SOURCE, "avg_launch_ms": k3_ms,
                   "launches_per_step": len(k3) / steps, "share_of_step": sum(k3) / ms_total if world == 1 else None}
    return roof, roof_k3


def conv_roofline(log, ms_total, steps, world):
    """Image branch "tcgen05": the slab convolutions (cp_conv_slab) of the timed loop against the sustained bf16 tensor peak.
    Flops are those of the convolutions proper (the border rows the kernel also multiplies are not counted)."""
    _, _, tf_sus, peak_src = load_peaks()
    cs = [(a.elapsed_time(b), sig[5]) for sig, a, b in log if sig[0] == "CS"]
    if not cs:
        return None
    ms = sum(t for t, _ in cs)
    flops = 2.0 * sum(m for _, m in cs)
    ach = flops / (ms * 1e-3) / 1e12
    return {"bound": "tensor", "kernel": "conv_slab_kernel (up_net 3x3 / transposed parities / patch_generator 2x2 / seg_block, bf16, all launches)",
            "achieved": ach, "peak": tf_sus, "unit": "TFLOP/s", "frac": ach / tf_sus, "peak_source": peak_src + ", sustained bf16",
            "launches_per_step": len(cs) / steps, "ms_per_step": ms / steps, "share_of_step": ms / ms_total if world == 1 else None}


def timed_loop(step, feats, steps, barrier, world, dev):
    """Exactly ``steps`` steps bracketed by barrier + synchronize on both sides; CUDA events; max over ranks (ms)."""
    import torch.distributed as dist
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    done = None
    for _ in range(steps):
        _, done = step(feats)
    torch.cuda.current_stream().wait_event(done)     # the last step's side-stream gather ends inside the timed region
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def run_ours(args):
    import torch.distributed as dist
    from checkerpose_b200 import _lib, build as cpbuild, dist as cpdist, head, ops

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback); use --impl reference for the CPU arm"
    assert os.path.realpath(_lib.LIB_PATH) == os.path.realpath(cpbuild.IN_TREE_LIB) and "CHECKERPOSE_B200_LIB" not in os.environ, \
        "bench.py measures the in-tree build of the library (unset CHECKERPOSE_B200_LIB)"
    torch.cuda.set_device(local)
    numa_bound = cpdist.bind_to_gpu_numa_node(local) if world > 1 else False   # before any pinned allocation
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    torch.set_grad_enabled(False)
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    head.set_compute_dtype(dtype)
    head.set_image_branch(args.image_branch)
    wl = workload(args, world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if wl["name"] == "lm_sweep":
        return run_sweep(args, wl, dev, rank, world, dtype, barrier)

    case = build_case(wl, dev, rank)
    B, N = case["B"], case["N"]
    feats, bbox = make_inputs(case, dev, dtype, rank)
    gather = cpdist.OverlappedGather(dev)
    last = {} if args.dump_outputs else None
    step = make_step(wl, case, bbox, gather, last)

    nwarm = args.warmup if args.profile else max(args.warmup, 3)
    for _ in range(nwarm):
        step(feats)
    barrier()

    # ---------------- timed region: inputs resident in HBM ----------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ops.chain_event_log = []
    n0 = ops.launch_count
    ms_total = timed_loop(step, feats, args.steps, barrier, world, dev)
    launches = ops.launch_count - n0
    log, ops.chain_event_log = ops.chain_event_log, None
    clocks = sampler.stop() if rank == 0 else None
    ms_step = ms_total / args.steps
    value = B * world / (ms_step * 1e-3)
    roof, roof_k3 = kernel_rooflines(log, ms_total, args.steps, B, N, dtype, world)
    roof_conv = conv_roofline(log, ms_total, args.steps, world)
    if last is not None and rank == 0:
        dump_outputs(args.dump_outputs, last)      # the last timed step's outputs, before the legs below run the step again

    if args.profile:   # under ncu: no e2e / CPU legs, numbers printed here are NOT bench values
        if rank == 0:
            print(json.dumps({"profile_run": True, "ms_per_step": ms_step, "gpu_launches": launches, "roofline": roof, "roofline_k3": roof_k3}))
        return

    # ---------------- GNN-only: the same step without the library convolutions of the image branch ----------------
    gnn_only = None
    if not wl["init_only"]:
        with head.reuse_image_branch():
            for _ in range(2):
                step(feats)
            ms_g = timed_loop(step, feats, args.steps, barrier, world, dev) / args.steps
        gnn_only = {"value": B * world / (ms_g * 1e-3), "unit": UNIT, "ms_per_step": ms_g,
                    "note": "up_net / patch_generator / seg_block outputs (the image branch) reused from a previous step of the same "
                            "batch; everything else (conv1x1 GEMM, K2, K3, query MLPs, decode, records) runs"}

    # ---------------- e2e: pinned host buffers -> public API -> host, every step ----------------
    host_feats = [f.cpu().pin_memory() for f in feats]
    dbuf = [[torch.empty_like(f) for f in feats] for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    h2d_bytes = sum(f.numel() * f.element_size() for f in feats)
    # rank 0 reads back ALL gathered records (it is the consumer of the gather); the other ranks read back their own shard
    out0, _ = step(feats)
    torch.cuda.synchronize()
    row_shape = tuple(out0.shape[1:])
    d2h_rows = B * world if (rank == 0 and not wl["init_only"]) else B
    host_out = [torch.empty((d2h_rows,) + row_shape, dtype=out0.dtype).pin_memory() for _ in range(2)]
    d2h_bytes = host_out[0].numel() * host_out[0].element_size()
    d2h_stream = torch.cuda.Stream(device=dev)

    def upload(i):
        s = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[s])
            for d, h in zip(dbuf[s], host_feats):
                d.copy_(h, non_blocking=True)
            ready[s].record(copy_stream)

    def e2e_run(nsteps):
        main = torch.cuda.current_stream()
        for s in range(2):
            consumed[s].record(main)
        upload(0)
        for i in range(nsteps):
            if i + 1 < nsteps:
                upload(i + 1)                       # overlap the next step's H2D with this step's compute
            main.wait_event(ready[i % 2])
            out, done = step(dbuf[i % 2])
            consumed[i % 2].record(main)
            # the records go to pinned host memory on their own stream (double-buffered), under the next step's compute
            with torch.cuda.stream(d2h_stream):
                d2h_stream.wait_event(done)
                out.record_stream(d2h_stream)
                src = out if (world == 1 or rank == 0 or wl["init_only"]) else out[rank * B:(rank + 1) * B]
                host_out[i % 2].copy_(src, non_blocking=True)
        torch.cuda.synchronize()                    # every step's records are on the host when the timed region ends

    e2e_run(2)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    e2e_run(args.steps)
    ev1.record()
    barrier()
    e2e_ms = ev0.elapsed_time(ev1)                      # e2e_run ends with a device-wide synchronize: all copies are done at ev1
    e2e_wall_ms = (time.perf_counter() - t0) * 1e3      # host wall clock of the same region, reported beside the event time
    if world > 1:
        t = torch.tensor([e2e_ms, e2e_wall_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms, e2e_wall_ms = float(t[0].item()), float(t[1].item())
    e2e_value = B * world * args.steps / (e2e_ms * 1e-3)

    # ---------------- parity sample + CPU baseline (rank 0, outside the timed regions) ----------------
    parity = cpu_base = None
    if rank == 0 and not wl["init_only"] and not args.no_parity:
        parity = parity_sample(wl, case, feats, bbox, dtype)
    if rank == 0 and world == 1 and not args.no_cpu_baseline and wl["name"] == "full4096":
        cores = os.cpu_count() or 1
        v, n, ms, kind = cpu_reference_rois_per_s(steps=8, warmup=1, N=N, rois_per_step=1, budget_s=20.0)
        cpu_base = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
                    "sample": f"{n} x 1 RoI of the same workload (N={N}) through "
                              f"{'the unmodified reference modules' if kind == 'reference' else 'oracle/'} on torch CPU fp32, {ms:.0f} ms each"}

    if rank == 0:
        print(json.dumps({
            "metric": METRIC if wl["name"] == "full4096" else f"RoIs/sec ({wl['name']})", "value": value, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": nwarm, "ms_per_step": ms_step, "higher_is_better": True, "scaling": wl["scaling"],
            "vs_baseline": None, "dtype": args.dtype if args.dtype == "bf16" else "f32 (split-bf16 x3 tensor-core GEMMs, fp32 storage)",
            "data": "synthetic",
            "config": {"workload": wl["text"], "name": wl["name"], "rois_per_gpu": B, "rois_total": B * world, "npoint": N, "graph_k": case["K"],
                       "objects": f"{wl['ds']}/{wl['objs'][0]}" if len(wl["objs"]) == 1 else f"{wl['ds']}: {len(wl['objs'])} graphs, selected per RoI",
                       "image_branch": ("included: our implicit-GEMM convolutions on tcgen05 (cp_conv_slab / cp_conv_bf16 / cp_gemm_x3), no library kernel"
                                        if (args.image_branch == "tcgen05" or args.dtype == "fp32") else "included (cuDNN, library part of the path)"),
                       "inputs": ("the 1024@8^2 HRNet map (all the init net reads, init.py:111-112)" if wl["init_only"] else
                                  "the three HRNet maps the head reads (256@32^2, 512@16^2, 1024@8^2); the 128@64^2 map is never read "
                                  "(pipeline.py:361,372) and is neither created nor uploaded"),
                       "l2": "inputs (0.23 GB/step) and intermediates (>1 GB) exceed the 126 MB L2; no explicit flush",
                       "collective": ("all_gather_into_tensor of the packed correspondence records (16 + 2N bytes per RoI) per step, on a side "
                                      "stream overlapped with the next step, complete inside the timed region") if world > 1 else "none (1 GPU)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "wall_ms_per_step": e2e_wall_ms / args.steps,
                    "note": "pinned host feature maps -> forward_with_correspondences(packed=True) -> pinned host records; next step's H2D and the "
                            "previous step's gather + D2H overlap compute on side streams; with N > 1 rank 0 reads back all gathered records "
                            "(d2h_bytes_per_step), the other ranks their own shard",
                    "numa_bound": numa_bound},
            "gpu_launches": launches, "clocks": clocks, "roofline": roof, "roofline_k3": roof_k3, "roofline_conv": roof_conv, "gnn_only": gnn_only,
            "parity": parity, "cpu_baseline": cpu_base,
        }))
    if world > 1:
        dist.destroy_process_group()


def run_sweep(args, wl, dev, rank, world, dtype, barrier):
    """BASELINE configs[4]: LM net, N x K sweep; one JSON line whose ``sweep`` key holds the table and whose ``value`` is
    the N=4096, K=20 entry."""
    import torch.distributed as dist
    from checkerpose_b200 import dist as cpdist, head
    Ns = [int(x) for x in args.sweep_n.split(",")]
    Ks = [int(x) for x in args.sweep_k.split(",")]
    table = []
    last = {} if args.dump_outputs else None
    for N in Ns:
        for K in Ks:
            if K > N:
                continue
            case = build_case(wl, dev, rank, N=N, K=K)
            feats, bbox = make_inputs(case, dev, dtype, rank)
            gather = cpdist.OverlappedGather(dev)
            step = make_step(wl, case, bbox, gather, last)
            for _ in range(max(args.warmup, 3)):
                step(feats)
            ms = timed_loop(step, feats, args.steps, barrier, world, dev) / args.steps
            plan = head.graph_ctx(case["net"].refine_net[0].pre_query_block[0]._knn, case["obj_ids"], case["B"], dev).plan
            table.append({"npoint": N, "graph_k": K, "ms_per_step": ms, "rois_per_s": case["B"] * world / (ms * 1e-3),
                          "staged_kernel": bool(plan.staged), "max_distinct_rows_per_tile": int(plan.max_unique)})
            del case, feats, step
            torch.cuda.empty_cache()
    if last is not None and rank == 0:
        dump_outputs(args.dump_outputs, last)      # the last timed step of the last (N, K) entry
    if rank == 0:
        head_entry = next((t for t in table if t["npoint"] == 4096 and t["graph_k"] == 20), table[-1])
        print(json.dumps({"metric": "RoIs/sec (lm_sweep)", "value": head_entry["rois_per_s"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                          "warmup": max(args.warmup, 3), "ms_per_step": head_entry["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
                          "config": {"workload": wl["text"], "name": "lm_sweep", "rois_per_gpu": wl["per_gpu"], "value_entry": "N=4096, K=20"},
                          "sweep": table}))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="full4096", choices=["full4096", "init64", "ycbv1024", "lm_sweep"])
    ap.add_argument("--batch", type=int, default=0, help="RoIs per GPU per step (ycbv1024: RoIs in total); 0 = the config's own")
    ap.add_argument("--npoint", type=int, default=0)
    ap.add_argument("--graph-k", type=int, default=0)
    ap.add_argument("--sweep-n", default="512,1024,2048,4096")
    ap.add_argument("--sweep-k", default="8,16,20,32,40")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--image-branch", default="tcgen05", choices=["tcgen05", "cudnn"], help="bf16 mode: whose convolutions run the image branch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--profile", action="store_true", help="short run for ncu: timed loop only, warm-up exactly --warmup")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32, under 64 MB)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
