#!/usr/bin/env python
"""bench.py — BEV queries/s of the attention-sampling hot path at BEVFormer-base shapes (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dist U|G] [--dtype f16|i8|f32] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W

A step = one pass of the hot path over one 6-camera frame of synthetic NuScenes-shaped input:
  N = 1 : one MultiScaleDeformableAttn call at BASELINE configs[2] (200x200 BEV, 6 cams, 4 levels, 8 heads, 4x8 points)
  N > 1 : the same frame on a (camera group x query tile) grid of ranks: one fused sampling launch per rank (bev_mask
          camera sum folded in) and one reduce-scatter of the BEV accumulator inside the camera group — our kernel over
          NVLink peer memory, or NCCL ("scaling": "strong"). Every line also carries `scaling_anchor`: the same fused
          step on ONE GPU (same work as N > 1), because the N = 1 headline is the plain plugin op.
Input distribution: G (camera-ring geometry, the NuScenes-shaped case north_star names) is the headline; the reference unit
test's uniform distribution U (every point of every camera in range: worst case) is measured in the same run and printed
as `worst_case_U` with its own roofline.
`value` is timed with inputs resident in HBM (CUDA events on the launching stream, barrier + synchronize on both sides,
max over ranks); `e2e` is the same call through the public Python operator with pinned HOST buffers (H2D of the step's
inputs and D2H of its result inside the timed region). `roofline` divides the ALGORITHMIC bytes of one launch
(SURVEY §8(d): every input read once, output written once) by the kernel's measured duration and by the measured HBM
peak of MEASURED_PEAKS.json. `cpu_baseline` / `--impl reference` time the reference's CPU algorithm
(multi_scale_deformable_attn_pytorch restated in oracle/msda.py — kind "port": the reference's Python file cannot
travel to the GPU box) on the host cores, on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
WORKLOAD = "base_sca"
WORKLOAD_TEXT = ("base_sca: MultiScaleDeformableAttn 200x200 BEV (40000 queries), 6 cams, 4 levels "
                 "[[116,200],[58,100],[29,50],[15,25]], 8 heads x 32 ch, 4x8 points (BASELINE configs[2])")
DUMP_QUERIES = 4096  # 6 cameras x 4096 queries x 8 heads x 32 channels in float32: 25 MB
DIST_TEXT = {"U": "U: reference unit-test distribution (all points in range, worst case)",
             "G": "G: camera-ring geometry (~1/6 of camera x query pairs visible)"}


def workload_config(dist, gpus=1, flush=False):
    """The `config` object BOTH arms print, built from the same arguments so that the driver's comparison sees one
    configuration: workload, input distribution, how L2 is treated between timed steps, and the parallelism."""
    return {"workload": WORKLOAD_TEXT, "distribution": DIST_TEXT[dist],
            "l2": "flushed between launches (256 MiB memset)" if flush else
                  "no flush: the step's inputs (590 MB fp16) are larger than the 126 MB L2",
            "parallelism": "1 GPU" if gpus <= 1 else f"camera-group x query-tile shard over {gpus} GPUs"}


def load_workloads():
    """bevformer_tensorrt_b200/workloads.py loaded BY PATH (it needs torch only). The reference arm generates its inputs
    through this so that its process never imports the product package and never maps the product's .so."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("b200_workloads_standalone",
                                                  os.path.join(ROOT, "bevformer_tensorrt_b200", "workloads.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[spec.name] = mod
    spec.loader.exec_module(mod)
    return mod


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dist", default="G", choices=["U", "G"],
                    help="input distribution (SURVEY §8(d) config 3). G = the NuScenes-shaped camera-ring geometry that "
                         "north_star names (headline); U = the reference unit test's uniform worst case (always reported "
                         "next to it, `worst_case_U`)")
    ap.add_argument("--dtype", default="f16", choices=["f16", "f32", "i8"])
    ap.add_argument("--f16-mode", type=int, default=None, help="0 exact fp32 FMA, 1 mixed FHFMA (library default)")
    ap.add_argument("--round1-kernel", action="store_true", help="run csrc/msda.cu instead of the second-generation path")
    ap.add_argument("--flush-l2", action="store_true", help="write a 256 MiB buffer between timed launches")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-repeats", type=int, default=3)
    ap.add_argument("--ref-queries", type=int, default=5000,
                    help="--impl reference: BEV queries per step (all 6 cameras each); bounded so K steps stay short")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip the same-box GPU baseline of the reference's kernels")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N>1: reduce-scatter inside the camera group by our NVLink peer-memory kernel, or by NCCL")
    ap.add_argument("--graph", action="store_true",
                    help="N>1: replay the two-launch step from a CUDA graph (two steps per graph) instead of eager launches; "
                         "measured equal at N = 2 (0.201 vs 0.194 ms), and a capture next to a live NCCL communicator hung "
                         "once at N = 4 on this image, so it is opt-in")
    ap.add_argument("--overlap", action="store_true",
                    help="N>1: overlapped step (peers' rows sampled first, pulled under the own-rows launch); measured slower")
    ap.add_argument("--no-autotune", action="store_true",
                    help="keep the library's default MSDA launch shape instead of letting bt.autotune_msda pick one on the "
                         "step's tensors during warm-up")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary (other distribution / INT8) legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="1 GPU: after the timed steps, write the output of the last one to DIR/msda_output.npy (float32; "
                         f"a fixed, seeded sample of {DUMP_QUERIES} BEV queries, every camera, head and channel)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def ncu_traffic(key):
    """DRAM bytes per launch measured by ncu for this kernel/config (profiles/ncu_traffic.json), or None."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(key)
    except Exception:
        return None


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples nvidia-smi SM clocks / throttle reasons while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")  # fmt: skip

    def __init__(self, index):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                o = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                    str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()  # fmt: skip
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(float(r[0])) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(self.rows[0][1])), "reasons": reasons,
                "samples": len(sm)}  # fmt: skip


# ---------------------------------------------------------------------------------------------------------------
# CPU baseline (the only place bench.py touches oracle/)
# ---------------------------------------------------------------------------------------------------------------
def cpu_baseline(cfg, dist, nq, repeats):
    """Same bounded sample as --impl reference: all cameras x `nq` of the BEV queries, all host threads."""
    from bevformer_tensorrt_b200.workloads import make_msda_inputs
    from oracle import msda as omsda

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    value, shapes, ref, off, logits = make_msda_inputs(cfg, dist, 0, torch.float32)
    nq = min(nq, cfg.num_query)
    r, o, w = ref[:, :nq].contiguous(), off[:, :nq].contiguous(), logits[:, :nq].contiguous()
    omsda.msda_torch_port(value, shapes, r[:, :256], o[:, :256], w[:, :256])  # warm-up on a slice
    times = []
    for _ in range(max(1, repeats)):
        t0 = time.perf_counter()
        omsda.msda_torch_port(value, shapes, r, o, w)
        times.append(time.perf_counter() - t0)
    t = sorted(times)[len(times) // 2]
    return {"value": nq / t, "unit": "BEV queries/s", "cores": cores, "kind": "port",
            "sample": f"all {cfg.batch} cameras x {nq} of {cfg.num_query} BEV queries, fp32, distribution {dist}, "
                      f"median of {len(times)} calls ({t:.3f} s/call), torch {torch.__version__} "
                      f"multi_scale_deformable_attn_pytorch restated (oracle/msda.py)"}  # fmt: skip


def run_reference(args):
    """The reference's CPU implementation of the path (multi_scale_deformable_attn_pytorch, det2trt/models/utils/
    trt_ops.py:4-85, restated in oracle/msda.py — kind "port") on all host cores. A step = ALL 6 cameras x a fixed slice
    of the 40000 BEV queries (bounded sample, ~2 s), so that --steps K --warmup W are honoured as given and the printed
    ms_per_step is the true duration of a step. Never imports the product package."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = load_workloads()
    from oracle import msda as omsda

    assert "bevformer_tensorrt_b200" not in sys.modules
    cfg = wl.CONFIGS[WORKLOAD]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    value, shapes, ref, off, logits = wl.make_msda_inputs(cfg, args.dist, 0, torch.float32)
    nq = min(cfg.num_query, args.ref_queries)
    r, o, w = ref[:, :nq].contiguous(), off[:, :nq].contiguous(), logits[:, :nq].contiguous()
    steps, warm = max(1, args.steps), max(0, args.warmup)
    for _ in range(warm):
        omsda.msda_torch_port(value, shapes, r, o, w)
    t0 = time.perf_counter()
    for _ in range(steps):
        omsda.msda_torch_port(value, shapes, r, o, w)
    dt = (time.perf_counter() - t0) / steps
    qps = nq / dt  # one BEV query spans all 6 cameras, and all 6 were processed
    sample = (f"each step = all {cfg.batch} cameras x {nq} of {cfg.num_query} BEV queries (bounded sample of the frame), "
              f"fp32, {steps} steps after {warm} warm-up, torch {torch.__version__} on {cores} host threads; "
              "multi_scale_deformable_attn_pytorch restated (oracle/msda.py)")
    print(json.dumps({
        "impl": "reference", "metric": "BEV queries/s (BEVFormer-base shapes)", "value": qps, "unit": "BEV queries/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.dist, args.gpus, args.flush_l2),
        "cpu_baseline": {"value": qps, "unit": "BEV queries/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": qps, "unit": "BEV queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))  # fmt: skip


def ref_gpu_baseline(cfg, host, dist, peak):
    """Same-box GPU baseline: the reference's OWN CUDA kernels (oracle/_ref = its .cu files compiled unmodified) timed on
    the same device tensors with the same CUDA-event method: ms_deformable_im2col_cuda<float>, <__half>, _h2 and
    _int8<float|__half2> (…Kernel.cu:1106-1218). Baseline only — nothing here is on the product path."""
    from oracle import REF_LIB
    from oracle import msda as omsda

    if not os.path.exists(REF_LIB):
        return {"unavailable": "oracle/_ref/libref_kernels.so not built (needs /root/reference at build time)"}
    from bevformer_tensorrt_b200.workloads import quantize_per_tensor

    rk = omsda.RefKernels()
    value, shapes, ref, off, logits = host
    out = {"what": "reference kernels of TensorRT/plugin/multi_scale_deformable_attn compiled unmodified for sm_100a, "
                   f"distribution {dist}, CUDA events, mean of 10 launches after 2 warm-up"}
    sh = shapes.cuda()

    def t(fn, n=10, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    for variant, td, eb in (("f32", torch.float32, 4), ("f16", torch.float16, 2), ("f16_h2", torch.float16, 2)):
        dev = [x.to(td).cuda() for x in (value, ref, off, logits)]
        ms = t(lambda: rk.msda(dev[0], sh, dev[1], dev[2], dev[3], variant=variant))
        out[f"ms_deformable_im2col_cuda_{variant}"] = {
            "kernel_ms": ms, "bev_queries_per_s": cfg.num_query / (ms * 1e-3),
            "roofline_frac": cfg.algorithmic_bytes(eb) / (ms * 1e-3) / 1e9 / peak}
        del dev
    vq, sv = quantize_per_tensor(value)
    oq, so = quantize_per_tensor(off)
    wq, sw = quantize_per_tensor(logits)
    for rdt, tag in ((torch.float32, "int8_float_ref"), (torch.float16, "int8_half2_ref")):
        dev = [vq.cuda(), ref.to(rdt).cuda(), oq.cuda(), wq.cuda()]
        ms = t(lambda: rk.msda_i8(dev[0], sv, sh, dev[1], dev[2], so, dev[3], sw, 1.6 / 127.0))
        out[f"ms_deformable_im2col_cuda_{tag}"] = {
            "kernel_ms": ms, "bev_queries_per_s": cfg.num_query / (ms * 1e-3),
            "roofline_frac": cfg.algorithmic_bytes(1, 4 if rdt == torch.float32 else 2) / (ms * 1e-3) / 1e9 / peak}
    torch.cuda.empty_cache()
    return out


# ---------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------
def make_op(dtype, tensors):
    """Returns (callable running one MSDA on device-resident tensors, elem_bytes, ref_bytes)."""
    import bevformer_tensorrt_b200 as bt
    from bevformer_tensorrt_b200.workloads import quantize_per_tensor

    value, shapes, ref, off, logits = tensors
    if dtype == "i8":
        vq, sv = quantize_per_tensor(value)
        oq, so = quantize_per_tensor(off)
        wq, sw = quantize_per_tensor(logits)
        sout = 1.6 / 127.0  # PTQ output scale (amax of the fp32 result on this distribution ~1.5)
        dev = [vq.cuda(), shapes.cuda(), ref.half().cuda(), oq.cuda(), wq.cuda()]
        return (lambda: bt.multi_scale_deformable_attn_int8(dev[0], sv, dev[1], dev[2], dev[3], so, dev[4], sw, sout)), 1, 2, dev
    td = torch.float16 if dtype == "f16" else torch.float32
    dev = [value.to(td).cuda(), shapes.cuda(), ref.to(td).cuda(), off.to(td).cuda(), logits.to(td).cuda()]
    return (lambda: bt.multi_scale_deformable_attn(*dev)), (2 if dtype == "f16" else 4), None, dev


def autotune_launch_shape(bt, dev, enabled=True):
    """The product's own tactic selection (bt.autotune_msda: every launch shape of the FP16 / FP32 plugin op is run on
    THESE tensors, checked bit for bit against the default shape and timed with CUDA events; the fastest identical one is
    made the process-wide setting). Runs before the warm-up, outside every timed region. Any failure falls back to the
    default shape and is reported in the line."""
    if not enabled:
        bt.set_msda_launch_shape("default")
        return {"chosen": "default", "note": "--no-autotune"}
    try:
        return bt.autotune_msda(*dev)
    except Exception as e:  # noqa: BLE001 — the bench must still produce its line on the default shape
        try:
            bt.set_msda_launch_shape("default")
        except Exception:  # noqa: BLE001
            pass
        return {"chosen": "default", "error": repr(e)}


def autotune_fused(bt, run, result, enabled=True):
    """bt.autotune_msda_fused for the fused spatial-cross-attention forms (default launch vs 2 CTAs per SM), with the same
    fall-back rule as autotune_launch_shape. Local launches only: safe per rank before a collective step."""
    if not enabled:
        bt.set_msda_gather_variant(0)
        return {"chosen": "default", "note": "--no-autotune"}
    try:
        return bt.autotune_msda_fused(run, result)
    except Exception as e:  # noqa: BLE001
        try:
            bt.set_msda_gather_variant(0)
        except Exception:  # noqa: BLE001
            pass
        return {"chosen": "default", "error": repr(e)}


def time_kernel(fn, steps, warmup, flush=None):
    """Per-launch CUDA-event timing on the launching stream. Returns (total ms over steps, per-launch ms list)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in evs:
        if flush is not None:
            flush.zero_()
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    per = [a.elapsed_time(b) for a, b in evs]
    return sum(per), per


def dump_outputs(out_dir, y):
    """Writes the plugin op's output y [cameras, queries, heads, channels] (what a caller of the timed path receives) for
    comparing two builds output for output. The whole tensor is 245 MB in float32, so the same seeded sample of
    queries is taken every run."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    q = torch.randperm(y.shape[1], generator=torch.Generator().manual_seed(0))[:DUMP_QUERIES].sort().values
    np.save(os.path.join(out_dir, "msda_output.npy"), y[:, q.to(y.device)].float().cpu().numpy())


def run_single(args, cfg, peak, peak_src):
    from bevformer_tensorrt_b200 import _lib
    from bevformer_tensorrt_b200.workloads import make_msda_inputs

    if args.f16_mode is not None:
        _lib.load().b200_msda_set_f16_mode(args.f16_mode)
    import bevformer_tensorrt_b200 as bt

    v2_on = not args.round1_kernel
    bt.set_msda_v2(v2_on)
    torch.cuda.set_device(0)
    host = make_msda_inputs(cfg, args.dist, 0, torch.float32)
    fn, eb, rb, dev = make_op(args.dtype, host)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda") if args.flush_l2 else None
    tune = autotune_launch_shape(bt, dev, not args.no_autotune) if args.dtype in ("f16", "f32") else None

    for _ in range(max(3, args.warmup)):
        fn()
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    with ClockSampler(0) as clk:
        t_wall0 = time.perf_counter()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        start.record()
        for _ in range(args.steps):
            if flush is not None:
                flush.zero_()
            if args.dump_outputs:
                last = fn()
            else:
                fn()
        end.record()
        torch.cuda.synchronize()
        total_ms = start.elapsed_time(end)
        launches = _lib.launch_count() - n0  # kernels of this library launched inside the timed region
        wall = time.perf_counter() - t_wall0
        # keep the GPU busy a little longer if the region was too short for nvidia-smi to sample it
        while time.perf_counter() - t_wall0 < 1.0:
            fn()
        torch.cuda.synchronize()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
        del last
    ms_step = total_ms / args.steps
    # per-launch duration of the dominant (only) kernel, measured live with events around each launch
    _, per = time_kernel(fn, min(args.steps, 50), 3, flush)
    per.sort()
    k_ms = sum(per) / len(per)
    alg = cfg.algorithmic_bytes(eb, rb)
    achieved = alg / (k_ms * 1e-3) / 1e9
    out = {
        "metric": "BEV queries/s (BEVFormer-base shapes)", "value": cfg.num_query / (ms_step * 1e-3),
        "unit": "BEV queries/s", "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": {"f16": "f16 storage, f32 index math + accumulate", "f32": "f32", "i8": "i8 storage, f32 math"}[args.dtype],
        "data": "synthetic",
        "config": workload_config(args.dist, 1, args.flush_l2),
        "gpu_launches": int(launches),
        "clocks": clk.summary(),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": ncu_traffic(f"{args.dtype}_{args.dist}"),
                     "traffic_source": "static: dram__bytes_read+write per launch from the committed ncu --set full "
                                       "capture of this kernel/config (profiles/ncu_traffic.json), not re-measured in this run",
                     "kernel": ("msda_pack_kernel + msda_i8p_kernel: the op's two launches, timed together (pack pre-pass "
                                "included in the denominator)") if args.dtype == "i8" and v2_on else "msda_gather_kernel",
                     "kernel_ms": k_ms, "kernel_ms_min": per[0],
                     "launch_shape": "%s: %d unit(s) per warp%s, gather variant %d (bt.MSDA_LAUNCH_SHAPES)"
                                     % ((tune or {}).get("chosen", "default"), bt.get_msda_batch_units()[0],
                                        ", grid-strided" if bt.get_msda_batch_units()[1] else "", bt.get_msda_gather_variant()),
                     "algorithmic_bytes": alg, "peak_source": peak_src},
        "wall_s": wall,
    }  # fmt: skip
    if tune is not None:
        out["autotune"] = dict(tune, what="bt.autotune_msda on this step's device tensors before the warm-up (the product's "
                                          "tactic selection, as a TensorRT builder times a plugin's tactics): median ms of "
                                          "every launch shape whose output equals the default shape's bit for bit; the "
                                          "fastest is used for the timed region, the e2e leg and nothing else is changed")
    return out, fn, dev, host


class stdout_to_stderr:
    """File-descriptor level redirect of stdout (fd 1) into stderr (fd 2) for the duration of the block — catches
    output written by native libraries (NCCL's banner), not only Python's print."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def run_e2e(args, cfg, host):
    """Public-API call with pinned host buffers: H2D of the step's inputs + kernel + D2H of the result, per step."""
    import bevformer_tensorrt_b200 as bt

    td = {"f16": torch.float16, "f32": torch.float32, "i8": torch.float16}[args.dtype]
    value, shapes, ref, off, logits = host
    # staging buffers from cudaHostAlloc (bt.empty_pinned): tensor.pin_memory() measured 40-49 GB/s on this box
    # depending on where its pages were first touched, cudaHostAlloc 55 GB/s every time (profiles/r01_micro_h2d_bw.json)
    pinned = []
    for t in (value, ref, off, logits):
        h = bt.empty_pinned(t.shape, td)
        h.copy_(t.to(td))
        pinned.append(h)
    shapes_d = shapes.cuda()
    out_host = bt.empty_pinned((cfg.batch, cfg.num_query, cfg.num_heads, cfg.channels), td)
    h2d = sum(t.numel() * t.element_size() for t in pinned)
    d2h = out_host.numel() * out_host.element_size()

    # The host-buffer entry of the package: per-camera pipelining of H2D / kernel / D2H over three streams
    # (bevformer_tensorrt_b200/host_pipeline.py). Every step copies all of its inputs in and its whole result out; steps
    # issued back to back overlap across the step boundary exactly as the cameras overlap inside a step. The clock
    # stops after the last byte of the last step's result is in host memory.
    pipe = bt.HostMSDA()

    def step():
        pipe(pinned[0], shapes, pinned[1], pinned[2], pinned[3], out=out_host)

    def serial_step():
        v, r, o, w = (t.cuda(non_blocking=True) for t in pinned)
        out = bt.multi_scale_deformable_attn(v, shapes_d, r, o, w)
        out_host.copy_(out, non_blocking=True)

    for _ in range(2):
        serial_step()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(args.e2e_steps):
        serial_step()
    b.record()
    torch.cuda.synchronize()
    serial_ms = a.elapsed_time(b) / args.e2e_steps

    import time

    def timed(n):
        """CUDA events on the current stream around n pipelined steps: the end event waits for all three pipeline
        streams; the wall clock between the same two points is returned as a cross-check."""
        cur = torch.cuda.current_stream()
        pipe.synchronize()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(cur)
        for _ in range(n):
            step()
        for s in (pipe.s_in, pipe.s_k, pipe.s_out):
            cur.wait_stream(s)
        e1.record(cur)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n, (time.perf_counter() - t0) * 1e3 / n

    for _ in range(2):
        step()
    ms, wall_ms = timed(args.e2e_steps)
    single_ms, _ = timed(1)  # one isolated step (fill + drain of the camera pipeline included)
    return {"value": cfg.num_query / (ms * 1e-3), "unit": "BEV queries/s", "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h, "ms_per_step": ms, "steps": args.e2e_steps,
            "ms_single_isolated_step": single_ms, "ms_per_step_single_stream": serial_ms, "ms_per_step_wall": wall_ms,
            "note": "HostMSDA: pinned host -> device copies of value/ref/offsets/logits + kernel + device -> pinned host "
                    "copy of out, pipelined per camera over 3 streams; CUDA events around the steps, the end event waits for all 3 streams"}  # fmt: skip


def time_graph(fn, n=40, warm=5):
    """Device time per call of a short op: `n` calls captured into one CUDA graph (the ops launch on torch's current stream
    through the C ABI, so they are capturable), CUDA events around one replay after a warm replay. Takes the host launch
    path (Python wrapper, ctypes, driver: ~10 us per launch) out of ops that are 15-100 us long; returns us per call."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(n):
            fn()
    g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n * 1e3


def other_ops_legs(hbm_peak_gbs):
    """The other two plugins of the path under the same clock (CUDA events around a CUDA-graph replay of 40 calls):
    grid sampler prev-BEV warp [1,256,200,200] (BASELINE configs[3]) FP16 / kCHW2 / INT8-kCHW4 against the HBM roofline
    (inputs 10-41 MB: L2-resident between launches, stated), DCNv2 R101 stage-3 layer [6,256,58,100] 3x3 FP16 / INT8
    against the measured SUSTAINED bf16 tensor peak (the one dense contraction on the path)."""
    import bevformer_tensorrt_b200 as bt
    from bevformer_tensorrt_b200.functions.grid_sampler import pack_chw

    pk = {}
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    tens = float(pk.get("bf16_tflops_sustained", 1400.0))
    tens_src = "measured bf16_tflops_sustained" if "bf16_tflops_sustained" in pk else "fallback 1400 TFLOP/s sustained"
    out = {}
    H = W = 200
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(1, 256, H, W, device="cuda", generator=g)
    th = 0.05
    ys, xs = torch.meshgrid(torch.linspace(-1, 1, H, device="cuda"), torch.linspace(-1, 1, W, device="cuda"), indexing="ij")
    grid = torch.stack([xs * 0.9988 - ys * th, xs * th + ys * 0.9988], 0)[None].contiguous() * 10

    def leg(fn, nbytes, note):
        us = time_graph(fn)
        return {"kernel_us": us, "algorithmic_bytes": nbytes, "hbm_frac": nbytes / (us * 1e-6) / 1e9 / hbm_peak_gbs,
                "note": note}

    l2note = ("CUDA-graph replay of 40 back-to-back calls; tensors are L2-resident between launches (smaller than the "
              "126 MB L2): an on-chip-warm device-time figure")
    xh, gh = x.half(), grid.half()
    out["grid_sampler_f16_base"] = leg(lambda: bt.grid_sampler(xh, gh, "bilinear", "zeros", False), 41120000, l2note)
    x2, g2 = pack_chw(xh, 2), gh.permute(0, 2, 3, 1).unsqueeze(1).contiguous()
    out["grid_sampler_f16_chw2_base"] = leg(lambda: bt.grid_sampler_chw2(x2, g2, 256, "bilinear", "zeros", False),
                                            41120000, l2note)
    xi = torch.randint(-127, 127, (1, 64, H, W, 4), dtype=torch.int8, device="cuda")
    gi = torch.zeros(1, 1, H, W, 4, dtype=torch.int8, device="cuda")
    gi[..., 0] = (grid[0, 0] * 12.7).round().clamp(-127, 127).to(torch.int8)
    gi[..., 1] = (grid[0, 1] * 12.7).round().clamp(-127, 127).to(torch.int8)
    out["grid_sampler_i8_chw4_base"] = leg(
        lambda: bt.grid_sampler_int8(xi, 0.03, gi, 10 / 127, 0.03, 256, "bilinear", "zeros", False), 20640000, l2note)

    xd = torch.randn(6, 256, 58, 100, device="cuda", generator=g)
    off = torch.randn(6, 18, 58, 100, device="cuda", generator=g) * 2
    mask = torch.sigmoid(torch.randn(6, 9, 58, 100, device="cuda", generator=g))
    w = torch.nn.Parameter(torch.randn(256, 256, 3, 3, device="cuda", generator=g).half() / 48, requires_grad=False)
    b = torch.randn(256, device="cuda", generator=g).half()
    flops = 2 * 256 * 2304 * 5800 * 6

    def dleg(fn, note):
        us = time_graph(fn)
        return {"kernel_us": us, "tflops": flops / (us * 1e-6) / 1e12, "tensor_frac": flops / (us * 1e-6) / 1e12 / tens,
                "peak_tflops": tens, "peak_source": tens_src, "note": note}

    a16 = [xd.half(), off.half(), mask.half()]
    out["dcn_f16_base"] = dleg(lambda: bt.modulated_deformable_conv2d(*a16, w, b, 1, 1, 1, 1, 1),
                               "plugin op on NCHW input; NCHW->NHWC pre-pass + fused tcgen05 implicit GEMM; packed weights cached (constant at inference)")
    xcl = a16[0].contiguous(memory_format=torch.channels_last)
    out["dcn_f16_base_channels_last"] = dleg(lambda: bt.modulated_deformable_conv2d(xcl, a16[1], a16[2], w, b, 1, 1, 1, 1, 1),
                                             "channels-last input consumed in place: the fused kernel only")
    xq = torch.randint(-127, 127, (6, 64, 58, 100, 4), dtype=torch.int8, device="cuda")
    wq = torch.randint(-127, 127, (256, 64, 3, 3, 4), dtype=torch.int8, device="cuda")
    oq = torch.randint(-127, 127, (6, 18, 58, 100), dtype=torch.int8, device="cuda")
    mq = torch.randint(0, 127, (6, 9, 58, 100), dtype=torch.int8, device="cuda")
    out["dcn_i8_base"] = dleg(lambda: bt.modulated_deformable_conv2d_int8(xq, 0.02, oq, 0.03, mq, 1 / 127, wq, 0.001, b, 0.05, 256,
                                                                          1, 1, 1, 1, 1),
                              "INT8 kCHW4 plugin op: pre-passes + fused tcgen05 kernel, one requantisation")
    return out


def run_multi(args, cfg, peak, peak_src):
    """N > 1: camera-group x query-tile grid (sharding.plan_grid). Every rank runs ONE fused sampling launch (its cameras x
    its query tile, bev_mask camera-sum folded in) and ONE exchange launch: the reduce-scatter of the BEV accumulator
    inside its camera group, by our own kernel over NVLink peer memory (--exchange peer, default) or by NCCL
    reduce_scatter (--exchange nccl, the library baseline). Every rank ends up owning the final rows of 1/N of the BEV
    queries (the consumer, output_proj, is query-parallel)."""
    import torch.distributed as dist

    import bevformer_tensorrt_b200 as bt
    from bevformer_tensorrt_b200 import _lib
    from bevformer_tensorrt_b200.sharding import GroupedSCASampler, plan_grid
    from bevformer_tensorrt_b200.workloads import bev_reference_points_cam, camera_ring_lidar2img, make_msda_inputs

    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    if os.environ.get("B200_BENCH_HANG_DUMP"):  # debugging aid: stack of every thread if the run is still going after N s
        import faulthandler

        faulthandler.dump_traceback_later(int(os.environ["B200_BENCH_HANG_DUMP"]), exit=True)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    td = torch.float16 if args.dtype != "f32" else torch.float32
    value, shapes, ref, off, logits = make_msda_inputs(cfg, args.dist, 0, td)
    if args.dist == "G":
        _, bev_mask = bev_reference_points_cam(cfg.bev_hw, camera_ring_lidar2img(cfg.batch))
    else:
        # distribution U has every sampling point of every camera in range, i.e. every camera "sees" every query: the
        # matching visibility weights are 1/6 everywhere, so N>1 does exactly the work of the N=1 fused step
        bev_mask = torch.full((cfg.batch, cfg.num_query, 1), 1.0 / cfg.batch)
    width = cfg.num_heads * cfg.channels
    plan = plan_grid(cfg.batch, cfg.num_query, world)
    shard = plan[rank]
    exchange = args.exchange
    smp = GroupedSCASampler(shard, width, bt.multi_scale_deformable_attn_sca, exchange=exchange, overlap=args.overlap).load(
        value, shapes, ref, off, logits, bev_mask.to(td), dev)
    ok = torch.ones(1, device=dev)
    try:
        smp.connect(plan, dev)
    except Exception as e:  # noqa: BLE001 — symmetric memory unavailable: every rank falls back to NCCL together
        print(f"[bench] rank {rank}: peer-memory window failed ({type(e).__name__}: {e}); using NCCL reduce_scatter", file=sys.stderr)
        ok.zero_()
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if ok.item() == 0:
        exchange = "nccl"
        smp = GroupedSCASampler(shard, width, bt.multi_scale_deformable_attn_sca, exchange="nccl").load(
            value, shapes, ref, off, logits, bev_mask.to(td), dev).connect(plan, dev)

    # launch shape of the fused sampling kernel, picked per rank on its own shard (local launches only, no collective inside)
    tune_scratch = torch.zeros(shard.q1 - shard.q0, width, device=dev)

    def tune_run():
        tune_scratch.zero_()
        smp.compute(tune_scratch)

    fused_tune = autotune_fused(bt, tune_run, lambda: tune_scratch, not args.no_autotune)
    my_variant = bt.get_msda_gather_variant()
    deep = torch.tensor([1.0 if fused_tune.get("chosen") == "deep_gather" else 0.0], device=dev)
    dist.all_reduce(deep, op=dist.ReduceOp.SUM)
    del tune_scratch

    for _ in range(max(3, args.warmup)):
        smp.step()
    torch.cuda.synchronize()
    # CUDA graph of the step (two consecutive steps per graph: the partial buffers alternate) — only with our own exchange
    # kernel: the step then contains no library collective, and its launch parameters never change
    graphed = False
    if smp.exchange == "peer" and args.graph:
        flag = torch.ones(1, device=dev)
        try:
            smp.capture_pair()
            smp.step_pair()
        except Exception as e:  # noqa: BLE001
            print(f"[bench] rank {rank}: CUDA-graph capture of the step failed ({type(e).__name__}: {e}); eager launches", file=sys.stderr)
            flag.zero_()
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        graphed = flag.item() == 1
    # ---- correctness of the sharded result on hardware: owned slices gathered on rank 0 vs the single-GPU fused op
    got = smp.step().float().clone()
    rows_max = max(x.own1 - x.own0 for x in plan)
    pad = torch.zeros(rows_max, width, device=dev)
    pad[: got.shape[0]] = got
    gathered = [torch.empty_like(pad) for _ in range(world)] if rank == 0 else None
    dist.gather(pad, gathered, dst=0)
    max_abs_vs_1gpu = anchor_ms = anchor_tune = None
    if rank == 0:
        full = [t.to(dev) for t in (value, shapes, ref, off, logits)]
        want = bt.multi_scale_deformable_attn_sca(*full, bev_mask.to(dev))
        err = 0.0
        for x, g in zip(plan, gathered):
            err = max(err, (g[: x.own1 - x.own0] - want[x.own_queries().to(dev)]).abs().max().item())
        max_abs_vs_1gpu = err
        # the same fused step on ONE GPU (same work as the sharded step), timed like the kernel legs of the N=1 run
        bm_d = bev_mask.to(dev)

        def one_gpu_step():
            want.zero_()
            bt.multi_scale_deformable_attn_sca(*full, bm_d, want)

        anchor_tune = autotune_fused(bt, one_gpu_step, lambda: want, not args.no_autotune)  # the anchor gets its own best shape
        _, per1 = time_kernel(one_gpu_step, 20, 3)
        anchor_ms = sum(per1) / len(per1)
        bt.set_msda_gather_variant(my_variant)  # back to the shape picked for this rank's shard
        del full, want, bm_d
    del value, ref, off, logits
    torch.cuda.empty_cache()

    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    with ClockSampler(local) as clk:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        if graphed:
            for _ in range((args.steps + 1) // 2):
                smp.step_pair()
        else:
            for _ in range(args.steps):
                smp.step()
        b.record()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / (2 * ((args.steps + 1) // 2) if graphed else args.steps)
        launches = _lib.launch_count() - n0
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < 0.7:
            smp.step()
        torch.cuda.synchronize()
    # breakdown (reported separately, SURVEY §8(d) config 5): the local sampling launch alone, the exchange alone
    scratch = torch.zeros(shard.q1 - shard.q0, width, device=dev)
    a2, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a2.record()
    for _ in range(20):
        smp.compute(scratch)
    b2.record()
    torch.cuda.synchronize()
    ms_compute = a2.elapsed_time(b2) / 20
    dist.barrier()
    a3, b3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a3.record()
    for _ in range(20):
        smp.exchange_only()
    b3.record()
    torch.cuda.synchronize()
    ms_exchange = a3.elapsed_time(b3) / 20
    # end to end: every step copies this rank's shard of the inputs from pinned host memory, runs the sharded step and
    # reads this rank's owned rows of the BEV accumulator back to pinned host memory
    pinned = [t.cpu().pin_memory() for t in smp.local]
    out_host = torch.empty_like(smp.out, device="cpu").pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in pinned)
    d2h = out_host.numel() * out_host.element_size()

    def e2e_step():
        for d_t, h_t in zip(smp.local, pinned):
            d_t.copy_(h_t, non_blocking=True)
        out_host.copy_(smp.step(), non_blocking=True)

    for _ in range(2):
        e2e_step()
    torch.cuda.synchronize()
    dist.barrier()
    a4, b4 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a4.record()
    for _ in range(args.e2e_steps):
        e2e_step()
    b4.record()
    torch.cuda.synchronize()
    dist.barrier()
    ms_e2e = a4.elapsed_time(b4) / args.e2e_steps
    t = torch.tensor([ms, ms_compute, ms_exchange, ms_e2e], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_compute, ms_exchange, ms_e2e = t.tolist()
    hb = torch.tensor([float(h2d), float(d2h)], device="cuda", dtype=torch.float64)
    dist.all_reduce(hb, op=dist.ReduceOp.SUM)
    h2d_total, d2h_total = int(hb[0].item()), int(hb[1].item())
    eb = 2 if td == torch.float16 else 4
    alg = cfg.algorithmic_bytes(eb)
    out = None
    if rank == 0:
        achieved = alg / (ms_compute * 1e-3) / 1e9 / world  # per-GPU share of the frame's algorithmic bytes
        out = {
            "metric": "BEV queries/s (BEVFormer-base shapes)", "value": cfg.num_query / (ms * 1e-3),
            "unit": "BEV queries/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f16 storage, f32 index math + accumulate" if eb == 2 else "f32", "data": "synthetic",
            "config": workload_config(args.dist, world, False),
            "sharding": {"camera_groups": shard.groups, "query_tiles": shard.tiles,
                         "tile_layout": (f"interleaved blocks of {shard.block} BEV queries (balances the visible (camera, query) "
                                         "pairs between the ranks of a camera group)") if shard.block else "contiguous query ranges",
                         "per_rank": f"{shard.cam1 - shard.cam0} cameras x {shard.q1 - shard.q0} queries, one fused "
                                     "sampling launch (bev_mask camera-sum folded in) into an fp32 partial accumulator",
                         "exchange": {"peer": "b200_sca_peer_reduce: reduce-scatter inside the camera group by our kernel over "
                                              "NVLink peer memory (torch symmetric-memory window); no NCCL call in the step",
                                      "nccl": "NCCL reduce_scatter_tensor on the camera group's communicator",
                                      "none": "no exchange (one camera group)"}[smp.exchange],
                         "result": f"every rank owns the final fp32 rows of {shard.own1 - shard.own0} BEV queries"},
            "max_abs_vs_1gpu": max_abs_vs_1gpu,
            "autotune": {"what": "bt.autotune_msda_fused per rank on its own shard before the warm-up (default launch vs 2 CTAs "
                                 "per SM with 16 tap loads in flight per warp; result checked against the default's)",
                         "rank0": fused_tune, "ranks_on_deep_gather": int(deep.item()), "scaling_anchor": anchor_tune},
            "launch_mode": ("CUDA graph replay, two steps per graph (sampling launch + exchange launch each)" if graphed
                            else "eager launches (two per step)"),
            "scaling_anchor": {"what": "the same fused step (all cameras, all queries, no exchange) on rank 0's GPU alone, "
                                       "measured in this run before the sharded loop: same work as this N-GPU step",
                               "ms_per_step": anchor_ms, "value": cfg.num_query / (anchor_ms * 1e-3), "unit": "BEV queries/s"},
            "gpu_launches": int(launches), "clocks": clk.summary(),
            "breakdown_ms": {"step": ms, "local_sampling_launch": ms_compute, "exchange_only": ms_exchange},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": None, "kernel": "msda_gather_kernel (per-GPU share, local compute only)",
                         "algorithmic_bytes": alg, "peak_source": peak_src},
            "e2e": {"value": cfg.num_query / (ms_e2e * 1e-3), "unit": "BEV queries/s", "h2d_bytes_per_step": h2d_total,
                    "d2h_bytes_per_step": d2h_total, "ms_per_step": ms_e2e, "steps": args.e2e_steps,
                    "note": "per rank: pinned host -> device copy of its shard (value, ref, offsets, logits, bev_mask) + "
                            "sharded step + device -> pinned host copy of the rows it owns"},
        }  # fmt: skip
    dist.destroy_process_group()
    return out


def main():
    args = parse()
    if args.impl == "reference":  # before anything of the product is imported
        run_reference(args)
        return
    from bevformer_tensorrt_b200.workloads import CONFIGS

    cfg = CONFIGS[WORKLOAD]
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device. The product path has no CPU fallback; run under gpurun.")
    peak, peak_src = hbm_peak()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1 and args.dump_outputs:
        raise SystemExit("bench.py: --dump-outputs writes the 1-GPU step's output; run it with --gpus 1")
    if world > 1:
        # NCCL prints its version banner to stdout at communicator creation when the box sets NCCL_DEBUG=VERSION; the
        # contract is ONE JSON line on stdout, so everything the run itself emits goes to stderr until the line is ready
        with stdout_to_stderr():
            out = run_multi(args, cfg, peak, peak_src)
        if out is not None:
            print(json.dumps(out), flush=True)
        return

    out, fn, dev, host = run_single(args, cfg, peak, peak_src)
    out["e2e"] = run_e2e(args, cfg, host)
    if not args.no_secondary:
        # the other distribution and the other precisions, same shapes, same timing method (explains the headline)
        sec = {}
        from bevformer_tensorrt_b200 import _lib

        import bevformer_tensorrt_b200 as bt

        # (dtype, distribution, second-generation path on?) — the *_round1_kernel legs run csrc/msda.cu on the same
        # tensors (A/B of the rework); f32 has only the round-1 kernel
        # (dtype, distribution, second-generation INT8 path on?) — the i8_*_round1_kernel legs run csrc/msda.cu's gather
        # kernel on the same INT8 tensors (A/B of the rework); FP16 / FP32 have one kernel
        for dtype, dist_name, v2 in (("f16", "U", True), ("f16", "G", True), ("i8", "U", True), ("i8", "G", True),
                                     ("i8", "U", False), ("i8", "G", False), ("f32", "U", True)):  # fmt: skip
            if dtype == args.dtype and dist_name == args.dist and v2:
                continue
            from bevformer_tensorrt_b200.workloads import make_msda_inputs

            h = make_msda_inputs(cfg, dist_name, 0, torch.float32)
            prev = bt.set_msda_v2(v2)
            f2, eb, rb, _d = make_op(dtype, h)
            leg_tune = autotune_launch_shape(bt, _d, not args.no_autotune) if dtype in ("f16", "f32") else None
            _, per = time_kernel(f2, 30, 5)
            bt.set_msda_v2(prev)
            k = sum(per) / len(per)
            alg = cfg.algorithmic_bytes(eb, rb)
            key = f"{dtype}_{dist_name}" + ("" if v2 else "_round1_kernel")
            sec[key] = {"kernel_ms": k, "bev_queries_per_s": cfg.num_query / (k * 1e-3),
                        "roofline_frac": alg / (k * 1e-3) / 1e9 / peak, "algorithmic_bytes": alg}
            if leg_tune is not None:
                sec[key]["autotune"] = leg_tune
            del f2, _d, h
            torch.cuda.empty_cache()
        # the other MSDA call sites of a BEVFormer-base frame (SURVEY §8(f)-2): temporal self-attention (2 x 40000 queries, one
        # 200x200 level, 4 points) and the decoder (900 queries), FP16, every point in range; short ops -> CUDA-graph replay
        from bevformer_tensorrt_b200.workloads import make_msda_inputs

        for cname in ("base_tsa", "base_decoder"):
            ccfg = CONFIGS[cname]
            h = make_msda_inputs(ccfg, "U", 0, torch.float32)
            f2, eb, rb, _d = make_op("f16", h)
            leg_tune = autotune_launch_shape(bt, _d, not args.no_autotune)
            us = time_graph(f2)
            alg = ccfg.algorithmic_bytes(eb, rb)
            sec[f"f16_{cname}"] = {"kernel_us": us, "algorithmic_bytes": alg, "rate_over_hbm_peak": alg / (us * 1e-6) / 1e9 / peak,
                                   "autotune": leg_tune,
                                   "note": "CUDA-graph replay of 40 calls; tensors mostly L2-resident between launches"}
            del f2, _d, h
            torch.cuda.empty_cache()
        # back to the headline's launch shape for everything that follows
        bt.set_msda_launch_shape((out.get("autotune") or {}).get("chosen", "default"))
        other = "U" if args.dist == "G" else "G"
        o = sec.get(f"{args.dtype}_{other}")
        if o is not None:
            out["worst_case_U" if other == "U" else "geometry_G"] = {
                "what": f"same op, same shapes, distribution {DIST_TEXT[other]}; per-launch CUDA events, mean of 30",
                "value": o["bev_queries_per_s"], "unit": "BEV queries/s", "ms_per_step": o["kernel_ms"],
                "roofline": {"bound": "hbm", "achieved": o["algorithmic_bytes"] / (o["kernel_ms"] * 1e-3) / 1e9, "peak": peak,
                             "unit": "GB/s", "frac": o["roofline_frac"], "traffic": ncu_traffic(f"{args.dtype}_{other}"),
                             "algorithmic_bytes": o["algorithmic_bytes"]}}
        # fused SCA sampling (MSDA + bev_mask camera-sum into the fp32 BEV accumulator; SURVEY §8(f)-1): what the
        # sharded N>1 path runs per rank, timed here on one GPU (includes zeroing the accumulator). Each distribution
        # gets ITS OWN visibility weights: U -> every camera sees every query (1/6 everywhere: the same sampling work as
        # the plugin op, this is the same-work N=1 anchor of the scaling curve); G -> the camera ring's bev_mask.
        from bevformer_tensorrt_b200.workloads import bev_reference_points_cam, camera_ring_lidar2img, make_msda_inputs

        _, ring = bev_reference_points_cam(cfg.bev_hw, camera_ring_lidar2img(cfg.batch))
        masks = {"U": torch.full((cfg.batch, cfg.num_query, 1), 1.0 / cfg.batch).cuda(), "G": ring.cuda()}
        for dist_name in ("U", "G"):
            h = [t.cuda() for t in make_msda_inputs(cfg, dist_name, 0, torch.float16)]
            bm = masks[dist_name]
            acc = torch.zeros(cfg.num_query, cfg.num_heads * cfg.channels, device="cuda")

            def fused():
                acc.zero_()
                bt.multi_scale_deformable_attn_sca(*h, bm, acc)

            tune_f = autotune_fused(bt, fused, lambda: acc, not args.no_autotune)
            _, per = time_kernel(fused, 30, 5)
            k = sum(per) / len(per)
            sec[f"f16_{dist_name}_fused_sca_{'uniform' if dist_name == 'U' else 'ring'}_mask"] = {
                "kernel_ms": k, "bev_queries_per_s": cfg.num_query / (k * 1e-3), "autotune": tune_f,
                "note": "zero the 41 MB fp32 accumulator + fused kernel; no per-camera output; "
                        + ("uniform 1/6 visibility = same sampling work as the plugin op (N=1 anchor of the scaling curve)"
                           if dist_name == "U" else "camera-ring bev_mask")}
            # camera-shared form: offsets / logits passed once (the reference repeats the query per camera, so the
            # plugin's six copies are identical), cameras looped in registers, one plain store per slot
            hs = [h[0], h[1], h[2], h[3][:1].contiguous(), h[4][:1].contiguous()]
            last = [None]

            def shared():
                last[0] = bt.multi_scale_deformable_attn_sca_shared(*hs, bm)

            tune_s = autotune_fused(bt, shared, lambda: last[0], not args.no_autotune)
            _, per = time_kernel(shared, 30, 5)
            k = sum(per) / len(per)
            sb = 2 * (h[0].numel() + h[2].numel() + hs[3].numel() + hs[4].numel()) + 4 * bm.numel() + 4 * acc.numel()
            sec[f"f16_{dist_name}_shared_sca"] = {"kernel_ms": k, "bev_queries_per_s": cfg.num_query / (k * 1e-3),
                                                  "algorithmic_bytes": sb,
                                                  "roofline_frac": sb / (k * 1e-3) / 1e9 / peak,
                                                  "autotune": tune_s,
                                                  "note": "offsets/logits once for all cameras; single kernel, no memset"}
            del h, hs, last
        bt.set_msda_launch_shape((out.get("autotune") or {}).get("chosen", "default"))  # the headline's launch shape again
        torch.cuda.empty_cache()
        anchor = sec.get(f"f16_{args.dist}_fused_sca_{'uniform' if args.dist == 'U' else 'ring'}_mask")
        if anchor is not None and args.dtype == "f16":
            out["scaling_anchor"] = {
                "what": "the step bench.py --gpus N>1 runs (fused sampling + bev_mask camera sum into the fp32 BEV accumulator, "
                        "zeroing included) on ONE GPU: same work at every N; the N=1 headline above is the plain plugin op",
                "ms_per_step": anchor["kernel_ms"], "value": anchor["bev_queries_per_s"], "unit": "BEV queries/s"}
        sec.update(other_ops_legs(peak))
        out["secondary"] = sec
    if not args.no_ref_gpu:
        del fn, dev
        torch.cuda.empty_cache()
        out["ref_gpu_baseline"] = ref_gpu_baseline(cfg, host, args.dist, peak)
    if not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(cfg, args.dist, args.ref_queries, args.cpu_repeats)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
