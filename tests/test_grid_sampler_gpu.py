"""GPU parity tests for the grid sampler (pytest -m gpu). Checkers: oracle/grid_sampler_oracle.c (the reference FP32
kernel restated), golden vectors from the reference Python binding and from the reference's CUDA kernels run on a B200.
Tolerances: FP32 1e-5; FP16 1e-3 + output rounding slack for |out| > 2 (bicubic overshoots); INT8 2e-2-style bound in
units of the output scale."""
import itertools
import os

import numpy as np
import pytest
import torch

import bevformer_tensorrt_b200 as bt
from bevformer_tensorrt_b200.functions.grid_sampler import pack_chw, unpack_chw
from bevformer_tensorrt_b200.workloads import quantize_per_tensor
from oracle import grid_sampler as ogs
from tests.helpers import (GOLDEN, check_digest, load_ref_kernels, make_grid_sampler_inputs, make_rotation_grid,
                           sample_index)

pytestmark = pytest.mark.gpu

MODES = list(itertools.product(["bilinear", "nearest", "bicubic"], ["zeros", "border", "reflection"], [False, True]))
IM = {"bilinear": 0, "nearest": 1, "bicubic": 2}
PM = {"zeros": 0, "border": 1, "reflection": 2}


@pytest.mark.parametrize("interp,pad,align", MODES)
def test_fp32_matches_oracle_all_modes(interp, pad, align):
    inp, grid = make_grid_sampler_inputs(2, 7, 11, 13, 23, 19, seed=5)
    want = ogs.grid_sample_2d(inp.numpy(), grid.numpy(), IM[interp], PM[pad], align)
    for fn in (bt.grid_sampler, bt.grid_sampler2):
        got = fn(inp.cuda(), grid.cuda(), interp, pad, align).cpu().numpy()
        assert got.shape == want.shape
        assert np.abs(got - want).max() < 1e-5, (interp, pad, align, np.abs(got - want).max())


@pytest.mark.parametrize("interp,pad,align", MODES)
def test_fp32_matches_reference_golden(interp, pad, align):
    z = np.load(os.path.join(GOLDEN, "grid_sampler_ref.npz"))
    inp, grid = make_grid_sampler_inputs(2, 6, 11, 13, 17, 19, seed=3)
    got = bt.grid_sampler(inp.cuda(), grid.cuda(), interp, pad, align).cpu().numpy()
    d = np.abs(got - z[f"{interp}_{pad}_{int(align)}"])
    if interp == "nearest":
        assert (d > 1e-6).mean() < 0.01
    else:
        assert d.max() < 3e-5


@pytest.mark.parametrize("interp,pad,align", [("bilinear", "zeros", False), ("bilinear", "border", True),
                                               ("nearest", "reflection", False), ("bicubic", "zeros", False)])  # fmt: skip
def test_fp16_and_chw2_match_oracle(interp, pad, align):
    inp, grid = make_grid_sampler_inputs(2, 7, 12, 14, 20, 22, seed=6)
    inp, grid = inp.half(), grid.half()
    want = ogs.grid_sample_2d(inp.float().numpy(), grid.float().numpy(), IM[interp], PM[pad], align)
    tol = 1e-3 + np.abs(want).max() * 2.0**-11  # fp16 output rounding grows with |out| (bicubic overshoot)
    got = bt.grid_sampler(inp.cuda(), grid.cuda(), interp, pad, align)
    assert got.dtype == torch.float16
    assert np.abs(got.float().cpu().numpy() - want).max() < tol
    # kCHW2 packed layout (…TRT2)
    g2 = grid.permute(0, 2, 3, 1).unsqueeze(1).contiguous()  # [N,1,Ho,Wo,2] = (x, y)
    out2 = bt.grid_sampler_chw2(pack_chw(inp, 2).cuda(), g2.cuda(), inp.shape[1], interp, pad, align)
    got2 = unpack_chw(out2.cpu(), inp.shape[1])
    assert torch.equal(got2, got.cpu())


@pytest.mark.parametrize("interp,pad,align", [("bilinear", "zeros", False), ("nearest", "border", False),
                                               ("bicubic", "reflection", True)])  # fmt: skip
def test_int8_chw4_matches_dequant_oracle(interp, pad, align):
    inp, grid = make_grid_sampler_inputs(2, 10, 12, 14, 20, 22, seed=7, span=12.0)
    iq, si = quantize_per_tensor(inp)
    gq, sg = quantize_per_tensor(grid)
    real = ogs.grid_sample_2d(iq.float().numpy() * si, gq.float().numpy() * sg, IM[interp], PM[pad], align)
    so = float(np.abs(real).max()) / 127.0
    g4 = torch.zeros(grid.shape[0], 1, grid.shape[2], grid.shape[3], 4, dtype=torch.int8)
    g4[:, 0, :, :, 0], g4[:, 0, :, :, 1] = gq[:, 0], gq[:, 1]
    out4 = bt.grid_sampler_int8(pack_chw(iq, 4).cuda(), si, g4.cuda(), sg, so, inp.shape[1], interp, pad, align)
    got = unpack_chw(out4.cpu(), inp.shape[1]).float().numpy() * so
    assert np.abs(got - real).max() <= 0.5 * so + 1e-6  # one requantisation: at most half an output step


def _tile_grid(kind, N, Ho, Wo, seed):
    """[-10, 10] grids: "rot" = a small rotation + shift (compact source windows: the TMA tile path), "wild" = the
    reference test's sweep far beyond the image plus noise (windows larger than shared memory: the per-tile fallback),
    "mixed" = rotation in one image, wild in the other."""
    g = torch.Generator().manual_seed(seed)
    rot = make_rotation_grid(Ho, Wo, 7.5, shift=(3.3, -2.1)).repeat(N, 1, 1, 1)
    ys, xs = torch.meshgrid(torch.linspace(-14, 14, Ho), torch.linspace(-14, 14, Wo), indexing="ij")
    wild = torch.stack([xs, ys], 0)[None].repeat(N, 1, 1, 1) + 2.0 * torch.randn(N, 2, Ho, Wo, generator=g)
    if kind == "rot":
        return rot.contiguous()
    if kind == "wild":
        return wild.contiguous()
    out = rot.clone()
    out[1:] = wild[1:]
    return out.contiguous()


@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("kind", ["rot", "wild", "mixed"])
@pytest.mark.parametrize("pad,align", [("zeros", False), ("border", True), ("reflection", False)])
def test_tile_path_is_bit_identical_to_generic_kernel(kind, pad, align, mode):
    """2-D bilinear at TMA-legal layouts (row pitch a multiple of 16 bytes): the opt-in tile kernel — source window staged
    in shared memory by bulk copies per row (mode 1) or one 2-D tensor copy per channel packet (mode 2,
    cp.async.bulk.tensor.2d with a 16-byte-aligned window origin), or its per-tile fallback — and the generic kernel
    evaluate the same index arithmetic and the same FMA sequence per element, so every format must agree bit for bit; FP32
    additionally against the oracle. Shapes leave partial tiles on both output axes and a partial channel block (37
    channels)."""
    N, C, Hi, Wi, Ho, Wo = 2, 37, 26, 40, 19, 45
    g = torch.Generator().manual_seed(11)
    inp = torch.randn(N, C, Hi, Wi, generator=g)
    grid = _tile_grid(kind, N, Ho, Wo, 12)
    lib = bt._lib.load()

    def both(fn):
        prev = lib.b200_grid_sample_set_tile_path(mode)
        try:
            a = fn()
            lib.b200_grid_sample_set_tile_path(0)
            b = fn()
        finally:
            lib.b200_grid_sample_set_tile_path(prev)
        return a, b

    a, b = both(lambda: bt.grid_sampler(inp.cuda(), grid.cuda(), "bilinear", pad, align))
    assert torch.equal(a, b)
    want = ogs.grid_sample_2d(inp.numpy(), grid.numpy(), 0, PM[pad], align)
    assert np.abs(a.cpu().numpy() - want).max() < 1e-5
    ih, gh = inp.half(), grid.half()
    a, b = both(lambda: bt.grid_sampler(ih.cuda(), gh.cuda(), "bilinear", pad, align))
    assert torch.equal(a, b)
    g2 = gh.permute(0, 2, 3, 1).unsqueeze(1).contiguous()
    a, b = both(lambda: bt.grid_sampler_chw2(pack_chw(ih, 2).cuda(), g2.cuda(), C, "bilinear", pad, align))
    assert torch.equal(a, b)
    iq, si = quantize_per_tensor(inp)
    gq, sg = quantize_per_tensor(grid)
    g4 = torch.zeros(N, 1, Ho, Wo, 4, dtype=torch.int8)
    g4[:, 0, :, :, 0], g4[:, 0, :, :, 1] = gq[:, 0], gq[:, 1]
    a, b = both(lambda: bt.grid_sampler_int8(pack_chw(iq, 4).cuda(), si, g4.cuda(), sg, 0.05, C, "bilinear", pad, align))
    assert torch.equal(a, b)


def test_sampling_indices_bit_exact_via_nearest():
    """Nearest mode on an index-valued image returns the sampled flat index itself: the device's source-index
    arithmetic is compared bit-exactly with the oracle's (and thereby the reference kernel's formulas)."""
    Hi, Wi = 37, 41
    img = torch.arange(Hi * Wi, dtype=torch.float32).view(1, 1, Hi, Wi) + 1.0
    _, grid = make_grid_sampler_inputs(1, 1, Hi, Wi, 64, 64, seed=8, span=11.0)
    for pad, align in itertools.product(["zeros", "border", "reflection"], [False, True]):
        want = ogs.grid_sample_2d(img.numpy(), grid.numpy(), 1, PM[pad], align)
        got = bt.grid_sampler(img.cuda(), grid.cuda(), "nearest", pad, align).cpu().numpy()
        assert np.array_equal(got, want), (pad, align)


def test_3d_matches_reference_golden():
    z = np.load(os.path.join(GOLDEN, "grid_sampler_ref.npz"))
    inp3, grid3 = make_grid_sampler_inputs(1, 3, 5, 6, 7, 8, seed=4, depth=(4, 5))
    for interp, pad, align in itertools.product(["bilinear", "nearest"], ["zeros", "border", "reflection"], [False, True]):
        got = bt.grid_sampler(inp3.cuda(), grid3.cuda(), interp, pad, align).cpu().numpy()
        d = np.abs(got - z[f"3d_{interp}_{pad}_{int(align)}"])
        if interp == "nearest":
            assert (d > 1e-6).mean() < 0.02
        else:
            assert d.max() < 3e-5, (interp, pad, align, d.max())


def test_base_shape_identity_and_shift_properties():
    """BEVFormer-base prev-BEV warp shape [1,256,200,200]: an identity grid reproduces the input exactly; a one-pixel
    shift grid reproduces the shifted input (zeros padding)."""
    H = W = 200
    x = torch.randn(1, 256, H, W, device="cuda")
    xs = (torch.arange(W, device="cuda", dtype=torch.float32) + 0.5) / W * 20 - 10
    ys = (torch.arange(H, device="cuda", dtype=torch.float32) + 0.5) / H * 20 - 10
    gy, gx = torch.meshgrid(ys, xs, indexing="ij")
    grid = torch.stack([gx, gy], 0)[None].contiguous()
    out = bt.grid_sampler(x, grid, "bilinear", "zeros", False)
    assert (out - x).abs().max().item() < 5e-4  # fp32 grid coordinates carry ~1e-5 px of rounding x image gradient
    grid_s = grid.clone()
    grid_s[:, 0] += 20.0 / W  # sample one pixel to the right
    out_s = bt.grid_sampler(x, grid_s, "bilinear", "zeros", False)
    assert (out_s[..., :-1] - x[..., 1:]).abs().max().item() < 5e-4
    assert out_s[..., -1].abs().max().item() < 5e-4  # weight of the out-of-image tap ~1 -> zeros padding
    # FP16 storage: an fp16 grid near +-10 has a resolution of 2^-7 (~0.08 px here), so compare with the oracle on the
    # fp16-rounded grid instead of with the un-warped image
    xh, gh = x[:, :8].half(), grid.half()
    want = ogs.grid_sample_2d(xh.float().cpu().numpy(), gh.float().cpu().numpy(), 0, 0, False)
    outh = bt.grid_sampler(xh, gh, "bilinear", "zeros", False)
    assert np.abs(outh.float().cpu().numpy() - want).max() < 1e-3 + np.abs(want).max() * 2.0**-11


# the reference's own CUDA kernels, run on a B200 (tests/golden/ref_kernels_grid_sampler.npz, make_golden_ref_kernels.py)
REFK = load_ref_kernels("grid_sampler")


@pytest.mark.parametrize("interp,pad,align", MODES)
def test_fp32_matches_reference_kernel(interp, pad, align):
    """Against the reference's grid_sample<float> on a fixed, seeded sample of the output elements."""
    inp, grid = make_grid_sampler_inputs(2, 5, 17, 19, 33, 31, seed=9)
    check_digest(REFK, "fp32", inp, grid)
    got = bt.grid_sampler(inp.cuda(), grid.cuda(), interp, pad, align).cpu().numpy().reshape(-1)
    want = REFK[f"fp32_{interp}_{pad}_{int(align)}"]
    assert np.abs(got[sample_index(got.size, 512)] - want).max() < 1e-5, (interp, pad, align)


def test_base_shape_fp16_config4_vs_oracle_and_reference_kernel():
    """BASELINE configs[3], FP16 leg: prev-BEV warp [1,256,200,200] through a rotation grid, bilinear / zeros /
    align_corners=False, every output element vs the CPU oracle (reference FP32 formulas, gridSamplerKernel.cu:666-795,
    on the fp16-rounded tensors); kLINEAR and kCHW2 entries; the reference's own __half kernel (:797-1080, coordinates
    in half precision) on the same tensors, run on a B200 (REFK), must not come closer to those formulas."""
    g = torch.Generator().manual_seed(21)
    x = torch.randn(1, 256, 200, 200, generator=g).half()
    grid = make_rotation_grid(200, 200, 3.7, (2.25, -1.5)).half()
    want = ogs.grid_sample_2d(x.float().numpy(), grid.float().numpy(), 0, 0, False)
    tol = 1e-3 + np.abs(want).max() * 2.0**-11
    xd, gd = x.cuda(), grid.cuda()
    got = bt.grid_sampler(xd, gd, "bilinear", "zeros", False)
    e = np.abs(got.float().cpu().numpy() - want).max()
    assert e < tol, e
    g2 = grid.permute(0, 2, 3, 1).unsqueeze(1).contiguous().cuda()
    out2 = bt.grid_sampler_chw2(pack_chw(x, 2).cuda(), g2, 256, "bilinear", "zeros", False)
    assert torch.equal(unpack_chw(out2.cpu(), 256), got.cpu())
    check_digest(REFK, "base_fp16", x, grid)
    e_ref = float(REFK["base_fp16_err"])
    print(f"\n[grid sampler base fp16] ours {e:.3e}  reference __half kernel {e_ref:.3e} (vs fp32 formulas)")
    assert e <= e_ref + 1e-6


def test_base_shape_int8_config4_vs_dequant_oracle_and_reference_kernel():
    """BASELINE configs[3], INT8 leg: kCHW4 int8 input [1,256,200,200] and grid with per-tensor scales; ours vs the
    fp32 formulas on the dequantised tensors (at most half an output step: one requantisation), next to the reference's
    grid_sample_int8 (gridSamplerKernel.cu:2010-2043, :1082-1268: weights quantised to int8 at 1/127, dp4a), run on a
    B200 (REFK)."""
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
    out4 = bt.grid_sampler_int8(x4, si, g4d, sg, so, 256, "bilinear", "zeros", False)
    got = unpack_chw(out4.cpu(), 256).float().numpy() * so
    e = np.abs(got - real).max()
    assert e <= 0.5 * so + 1e-6, (e, so)
    check_digest(REFK, "base_int8", iq, gq)
    assert so == float(REFK["base_int8_so"])
    e_ref = float(REFK["base_int8_err"])
    print(f"\n[grid sampler base int8] ours {e / so:.3f} LSB  reference grid_sample_int8 {e_ref / so:.3f} LSB")
    # the reference kernel quantises its bilinear weights to int8 (x127) and requantises twice (:1137-1204): measured
    # ~30 output steps away from the fp32 formulas at this shape; ours carries the one final rounding
    assert e <= e_ref + 1e-6


@pytest.mark.parametrize("interp,pad,align", [("bilinear", "zeros", False), ("bilinear", "border", True), ("bicubic", "zeros", False)])
def test_backward_matches_the_reference_binding(interp, pad, align):
    """functions/grid_sampler.py:39-55: the input gradient equals autograd's of the reference binding's forward (its
    torch restatement in oracle/grid_sampler.py); the grid gradient is the REFERENCE's: its backward() returns ATen's
    gradient w.r.t. grid/10 multiplied by 10 (:55) where the chain rule gives a division — i.e. 100 x autograd's. The
    drop-in reproduces the reference's statement, so that is what is asserted."""
    inp, grid = make_grid_sampler_inputs(2, 5, 9, 11, 13, 12, seed=31, span=9.0)
    a, g = inp.cuda().requires_grad_(True), grid.cuda().requires_grad_(True)
    out = bt.grid_sampler(a, g, interp, pad, align)
    w = torch.randn_like(out)
    (out * w).sum().backward()
    a2, g2 = inp.cuda().requires_grad_(True), grid.cuda().requires_grad_(True)
    ref = ogs.grid_sampler_torch_port(a2, g2, IM[interp], PM[pad], align)
    (ref * w).sum().backward()
    assert (out - ref).abs().max().item() < 1e-5
    assert (a.grad - a2.grad).abs().max().item() < 1e-5 and (g.grad - 100 * g2.grad).abs().max().item() < 1e-2
    inp3, grid3 = make_grid_sampler_inputs(1, 3, 5, 6, 7, 8, seed=32, depth=(4, 5), span=9.0)
    a, g = inp3.cuda().requires_grad_(True), grid3.cuda().requires_grad_(True)
    (bt.grid_sampler(a, g, "bilinear", "zeros", False) ** 2).sum().backward()
    a2, g2 = inp3.cuda().requires_grad_(True), grid3.cuda().requires_grad_(True)
    (ogs.grid_sampler_torch_port(a2, g2, 0, 0, False) ** 2).sum().backward()
    assert (a.grad - a2.grad).abs().max().item() < 1e-4 and (g.grad - 100 * g2.grad).abs().max().item() < 1e-1


def test_error_behaviour():
    inp, grid = make_grid_sampler_inputs(1, 2, 4, 4, 5, 5)
    with pytest.raises(RuntimeError):
        bt.grid_sampler(inp, grid, "bilinear", "zeros", False)  # CPU tensor
    with pytest.raises(KeyError):
        bt.grid_sampler(inp.cuda(), grid.cuda(), "lanczos", "zeros", False)
    with pytest.raises(ValueError):
        bt.grid_sampler(inp.cuda(), grid.cuda()[:, :1], "bilinear", "zeros", False)
