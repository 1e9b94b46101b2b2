#!/usr/bin/env python
"""Fixtures from the reference's OWN CUDA kernels (oracle/_ref/libref_kernels.so: its .cu files compiled unmodified for
sm_100a by `make -C oracle ref`), for the GPU tests that compare this library with them:

    python tests/golden/make_golden_ref_kernels.py OUT_DIR [msda|grid_sampler|rotate|dcn ...]   # on a B200

writes OUT_DIR/ref_kernels_{msda,grid_sampler,rotate,dcn}.npz (all four unless some are named), which are committed
under tests/golden/. Each entry is keyed by the test case. Inputs are the tests' own seeded CPU inputs; `<case>_digest` is the SHA-256 of those inputs,
so a test can tell when its generator no longer reproduces them. Outputs too large for a fixture are stored as a fixed,
seeded sample (tests.helpers.sample_index), bit-exact comparisons as the SHA-256 of the whole output, and comparisons
that only need the reference's distance from a truth (its max-abs or mean-abs error) as that number, computed here over
every element.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bevformer_tensorrt_b200 as bt  # noqa: E402
from bevformer_tensorrt_b200.functions.grid_sampler import pack_chw, unpack_chw  # noqa: E402
from bevformer_tensorrt_b200.workloads import CONFIGS, MSDAConfig, make_msda_inputs, quantize_per_tensor  # noqa: E402
from oracle import REF_LIB  # noqa: E402
from oracle import dcn as odcn  # noqa: E402
from oracle import grid_sampler as ogs  # noqa: E402
from oracle import msda as omsda  # noqa: E402
from oracle import rotate as orot  # noqa: E402
from tests.helpers import (DCN_CASES, input_digest, make_dcn_inputs, make_grid_sampler_inputs,  # noqa: E402
                           make_rotation_grid, sample_index)

MSDA_FP32_CASES = [("small_sca", "edge", 71), ("tiny_sca", "U", 72), ("tsa_like", "U", 73)]
TSA_LIKE = MSDAConfig("tsa_like", 2, 1000, 8, 32, ((30, 30),), 4, 1)
ROTATE_CASES = [((8, 50, 50), 1.7, (25.0, 25.0)), ((7, 33, 47), 127.3, (20.5, 13.25)),
                ((256, 200, 200), -3.3, (100.0, 100.0)), ((32, 512, 512), 217.9, (500.0, 500.0))]
GS_MODES = [(i, p, a) for i in ("bilinear", "nearest", "bicubic") for p in ("zeros", "border", "reflection")
            for a in (False, True)]
IM = {"bilinear": 0, "nearest": 1, "bicubic": 2}
PM = {"zeros": 0, "border": 1, "reflection": 2}


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _sample(t, k, seed=0):
    flat = t.reshape(-1)
    idx = torch.from_numpy(sample_index(flat.numel(), k, seed)).to(flat.device)
    return flat[idx].cpu().numpy()


def _device():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name(0)


def msda():
    rk = omsda.RefKernels()
    z = {}
    for name, dist, seed in MSDA_FP32_CASES:
        inputs = make_msda_inputs(CONFIGS.get(name) or TSA_LIKE, dist, seed, torch.float32)
        key = f"fp32_{name}_{dist}_{seed}"
        z[f"{key}_digest"] = input_digest(*inputs)
        z[key] = _sample(rk.msda(*[t.cuda() for t in inputs], variant="f32"), 2048)
    base = CONFIGS["base_sca"]
    inputs = make_msda_inputs(base, "U", 0, torch.float32)
    z["fp32_base_U_0_digest"] = input_digest(*inputs)
    z["fp32_base_U_0"] = _sample(rk.msda(*[t.cuda() for t in inputs], variant="f32"), 4096)
    del inputs
    for dist in ("U", "G"):
        h = make_msda_inputs(base, dist, 1, torch.float16)
        hin = [t.cuda() for t in h]
        fin = [t.float() if t.is_floating_point() else t for t in hin]
        truth = rk.msda(*fin, variant="f32")
        z[f"fp16_base_{dist}_1_digest"] = input_digest(*h)
        z[f"fp16_base_{dist}_1_truth"] = _sample(truth, 2048)
        for variant in ("f16", "f16_h2"):  # reported next to ours by the test
            z[f"fp16_base_{dist}_1_err_{variant}"] = (rk.msda(*hin, variant=variant).float() - truth).abs().max().item()
        del hin, fin, truth
    for ref_dtype in (torch.float32, torch.float16):
        tag = str(ref_dtype).split(".")[-1]
        value, shapes, ref, off, logits = make_msda_inputs(CONFIGS["small_sca"], "U", 81, torch.float32)
        vq, sv = quantize_per_tensor(value)
        oq, so = quantize_per_tensor(off)
        wq, sw = quantize_per_tensor(logits)
        ref = ref.to(ref_dtype)
        real = omsda.msda_f32(vq.float().numpy() * sv, shapes.numpy(), ref.float().numpy(), oq.float().numpy() * so,
                              wq.float().numpy() * sw)  # fmt: skip
        sout = float(np.abs(real).max()) / 127.0
        theirs = rk.msda_i8(vq.cuda(), sv, shapes.cuda(), ref.cuda(), oq.cuda(), so, wq.cuda(), sw, sout)
        key = f"i8_small_sca_U_81_{tag}"
        z[f"{key}_digest"] = input_digest(vq, shapes, ref, oq, wq)
        z[f"{key}_sout"] = sout
        z[f"{key}_err"] = float(np.abs(theirs.cpu().numpy().astype(np.float32) * sout - real).max())
        z[key] = _sample(theirs, 4096)
    for dist in ("U", "G"):
        value, shapes, ref0, off, logits = make_msda_inputs(base, dist, 3, torch.float32)
        vq, sv = quantize_per_tensor(value)
        oq, so = quantize_per_tensor(off)
        wq, sw = quantize_per_tensor(logits)
        del value, off, logits
        for ref_dtype in (torch.float32, torch.float16):
            tag = str(ref_dtype).split(".")[-1]
            ref = ref0.to(ref_dtype)
            dq = [vq.cuda().float() * sv, shapes.cuda(), ref.cuda().float(), oq.cuda().float() * so, wq.cuda().float() * sw]
            truth = rk.msda(*dq, variant="f32")
            amax = truth.abs().max().item()
            sout = amax / 127.0
            theirs = rk.msda_i8(vq.cuda(), sv, shapes.cuda(), ref.cuda(), oq.cuda(), so, wq.cuda(), sw, sout)
            key = f"i8_base_{dist}_3_{tag}"
            z[f"{key}_digest"] = input_digest(vq, shapes, ref, oq, wq)
            z[f"{key}_truth_amax"] = amax
            z[f"{key}_err"] = (theirs.float() * sout - truth).abs().max().item()
            z[f"{key}_truth"] = _sample(truth, 2048)
            del dq, truth, theirs
            torch.cuda.empty_cache()
    return z


def grid_sampler():
    lib = ctypes.CDLL(REF_LIB)
    dims = lambda *s: (ctypes.c_int * 4)(*s)  # noqa: E731
    P = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    z = {}
    inp, grid = make_grid_sampler_inputs(2, 5, 17, 19, 33, 31, seed=9)
    z["fp32_digest"] = input_digest(inp, grid)
    inp, grid = inp.cuda(), grid.cuda()  # alive until the launches have run
    for interp, pad, align in GS_MODES:
        out = torch.empty(2, 5, 33, 31, device="cuda")
        lib.ref_grid_sample(0, P(out), P(inp), P(grid), dims(*out.shape), dims(*inp.shape), dims(*grid.shape), 4,
                            IM[interp], PM[pad], int(align), _stream())  # fmt: skip
        torch.cuda.synchronize()
        z[f"fp32_{interp}_{pad}_{int(align)}"] = _sample(out, 512)
    # BASELINE configs[3] FP16 leg: the reference's __half kernel, max-abs vs the FP32 formulas on the same tensors
    g = torch.Generator().manual_seed(21)
    x = torch.randn(1, 256, 200, 200, generator=g).half()
    grid = make_rotation_grid(200, 200, 3.7, (2.25, -1.5)).half()
    want = ogs.grid_sample_2d(x.float().numpy(), grid.float().numpy(), 0, 0, False)
    xd, gd = x.cuda(), grid.cuda()
    theirs = torch.empty(1, 256, 200, 200, dtype=torch.float16, device="cuda")
    lib.ref_grid_sample(1, P(theirs), P(xd), P(gd), dims(*theirs.shape), dims(*xd.shape), dims(*gd.shape), 4, 0, 0, 0,
                        _stream())  # fmt: skip
    torch.cuda.synchronize()
    z["base_fp16_digest"] = input_digest(x, grid)
    z["base_fp16_err"] = float(np.abs(theirs.float().cpu().numpy() - want).max())
    # INT8 leg: grid_sample_int8 on the quantised kCHW4 tensors, max-abs vs the FP32 formulas on the dequantised ones
    g = torch.Generator().manual_seed(22)
    x = torch.randn(1, 256, 200, 200, generator=g)
    grid = make_rotation_grid(200, 200, -2.9, (-1.75, 3.0))
    iq, si = quantize_per_tensor(x)
    gq, sg = quantize_per_tensor(grid)
    real = ogs.grid_sample_2d(iq.float().numpy() * si, gq.float().numpy() * sg, 0, 0, False)
    so = float(np.abs(real).max()) / 127.0
    g4 = torch.zeros(1, 1, 200, 200, 4, dtype=torch.int8)
    g4[:, 0, :, :, 0], g4[:, 0, :, :, 1] = gq[:, 0], gq[:, 1]
    x4, g4d = pack_chw(iq, 4).cuda(), g4.cuda()
    theirs4 = torch.empty(x4.shape, dtype=torch.int8, device="cuda")
    lib.ref_grid_sample_int8(P(theirs4), ctypes.c_float(so), P(x4), ctypes.c_float(si), P(g4d), ctypes.c_float(sg),
                             dims(1, 256, 200, 200), dims(1, 256, 200, 200), dims(1, 2, 200, 200), 4, 0, 0, 0, _stream())
    torch.cuda.synchronize()
    z["base_int8_digest"] = input_digest(iq, gq)
    z["base_int8_so"] = so
    z["base_int8_err"] = float(np.abs(unpack_chw(theirs4.cpu(), 256).float().numpy() * so - real).max())
    return z


def rotate():
    rr = orot.RefRotate()
    z = {}
    for shape, ang, ctr in ROTATE_CASES:
        g = torch.Generator().manual_seed(11)
        img = torch.randn(*shape, generator=g)
        angle, center = torch.tensor([ang]), torch.tensor(list(ctr))
        key = "x".join(map(str, shape))
        z[f"fp32_{key}_digest"] = input_digest(img, angle, center)
        for interp in ("bilinear", "nearest"):
            want = rr.rotate(img.cuda(), angle.cuda(), center.cuda(), IM[interp], "f32")
            torch.cuda.synchronize()
            if interp == "nearest":  # compared bit for bit: the whole output's digest
                z[f"fp32_{key}_nearest"] = input_digest(want.cpu())
            else:
                z[f"fp32_{key}_bilinear"] = _sample(want, 2048)
    # the reference's __half kernel: mean-abs distance from the FP32 formulas
    g = torch.Generator().manual_seed(3)
    img = torch.randn(16, 200, 200, generator=g)
    angle, center = torch.tensor([3.3]), torch.tensor([100.0, 100.0])
    truth = orot.rotate(img.half().float().numpy(), float(angle.half().float()[0]), center.numpy(), 0)
    theirs = rr.rotate(img.half().cuda(), angle.half().cuda(), center.half().cuda(), 0, "f16")
    torch.cuda.synchronize()
    z["fp16_digest"] = input_digest(img)
    z["fp16_mean_err"] = float(np.abs(theirs.float().cpu().numpy() - truth).mean())

    # device time per call of rotateKernel<float|__half> at BEVFormer-base size (same method as the test)
    def timed(fn, n=20):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n * 1e3

    g = torch.Generator().manual_seed(2)
    img = torch.randn(256, 200, 200, generator=g).cuda()
    angle, center = torch.tensor([2.3]).cuda(), torch.tensor([100.0, 100.0]).cuda()
    for tag, x, a, c in (("f32", img, angle, center), ("f16", img.half(), angle.half(), center.half())):
        z[f"time_reference_{tag}_us"] = min(timed(lambda: rr.rotate(x, a, c, 0, tag)) for _ in range(5))
        z[f"time_b200_{tag}_us"] = min(timed(lambda: bt.rotate(x, a, c, "bilinear")) for _ in range(5))
    z["time_device"] = _device()
    return z


def dcn():
    lib = ctypes.CDLL(REF_LIB)
    P = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    z = {}
    for case in ("k3_s1_p1_g2_dg2", "backbone_like"):
        x, off, mask, w, b, kw = make_dcn_inputs(case)
        N, Ci, H, W, Co, kh, kwid, s, p, d, g, dg = DCN_CASES[case]
        xs = [t.cuda() for t in (x, off, mask, w, b)]
        Ho, Wo = odcn.out_size(H, W, kh, kwid, s, p, d)
        out = torch.empty(N, Co, Ho, Wo, device="cuda")
        ws = torch.empty(Ci * kh * kwid * Ho * Wo + 64, device="cuda")
        lib.ref_dcn(0, P(xs[0]), P(xs[3]), P(xs[4]), P(xs[1]), P(xs[2]), P(out), P(ws), N, Ci, H, W, Co, kwid, kh, s, s,
                    p, p, d, d, g, dg, min(N, 32), _stream())  # fmt: skip
        torch.cuda.synchronize()
        z[f"fp32_{case}_digest"] = input_digest(x, off, mask, w, b)
        z[f"fp32_{case}_amax"] = out.abs().max().item()
        z[f"fp32_{case}"] = _sample(out, 2048)
    return z


def main(out_dir, names):
    os.makedirs(out_dir, exist_ok=True)
    device = _device()
    for name, fn in (("msda", msda), ("grid_sampler", grid_sampler), ("rotate", rotate), ("dcn", dcn)):
        if names and name not in names:
            continue
        z = fn()
        z["device"] = device
        np.savez_compressed(os.path.join(out_dir, f"ref_kernels_{name}.npz"), **z)
        print(name, {k: v for k, v in z.items() if np.ndim(v) == 0})


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2:])
