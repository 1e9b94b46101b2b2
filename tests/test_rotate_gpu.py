"""GPU parity tests for RotateTRT / RotateTRT2 (pytest -m gpu). Checkers: oracle/rotate_oracle.c (the reference FP32
kernel restated), golden vectors from the reference Python binding and from the reference's CUDA kernels run on a B200.
Tolerances: source indices bit-exact (given the device's cos/sin); FP32 values 1e-4 against the libm-trig oracle and
1e-6 against the reference kernel; FP16 1e-3 + output rounding; INT8 half an output step."""
import ctypes
import math
import os

import numpy as np
import pytest
import torch

import bevformer_tensorrt_b200 as bt
from bevformer_tensorrt_b200 import _lib
from bevformer_tensorrt_b200.functions.grid_sampler import pack_chw, unpack_chw
from bevformer_tensorrt_b200.workloads import quantize_per_tensor
from oracle import rotate as orot
from tests.helpers import (GOLDEN, ROTATE_CASES, check_digest, input_digest, load_ref_kernels, make_rotate_inputs,
                           sample_index)

pytestmark = pytest.mark.gpu

IM = {"bilinear": 0, "nearest": 1}
EXACT_HALF = ("right_angle",)  # source indices sit on x.5: a 1-ulp difference in cos/sin flips "nearest"


def device_trig(angle_deg):
    """cos/sin of the rotation as the device computes them (torch's float32 cos/sin are CUDA's cosf/sinf)."""
    ang = np.float32(np.float64(-np.float32(angle_deg)) * math.pi / 180.0)
    t = torch.tensor([ang], dtype=torch.float32, device="cuda")
    return float(torch.cos(t)[0]), float(torch.sin(t)[0])


def debug_indices(angle, center, H, W):
    out = torch.empty(H, W, 2, dtype=torch.float32, device="cuda")
    angle, center = angle.cuda(), center.cuda()  # keep both alive across the launch
    st = _lib.load().b200_rotate_debug_indices(angle.data_ptr(), center.data_ptr(),
                                               (ctypes.c_int * 3)(1, H, W), out.data_ptr(),
                                               _lib.current_stream_ptr())  # fmt: skip
    _lib.check("b200_rotate_debug_indices", st)
    return out.cpu().numpy()


@pytest.mark.parametrize("case", list(ROTATE_CASES))
def test_source_indices_bit_exact(case):
    C, H, W, ang, ctr = ROTATE_CASES[case]
    _, angle, center = make_rotate_inputs(case)
    got = debug_indices(angle, center, H, W)
    want = orot.source_indices(ang, ctr, H, W, trig=device_trig(ang))
    assert np.array_equal(got, want), np.abs(got - want).max()
    # and within rounding of the libm-trig oracle
    assert np.abs(got - orot.source_indices(ang, ctr, H, W)).max() < 1e-4


@pytest.mark.parametrize("case", list(ROTATE_CASES))
@pytest.mark.parametrize("interp", ["bilinear", "nearest"])
def test_fp32_matches_oracle(case, interp):
    img, angle, center = make_rotate_inputs(case)
    ang = ROTATE_CASES[case][3]
    for fn in (bt.rotate, bt.rotate2):
        got = fn(img.cuda(), angle.cuda()[0], center.cuda(), interp).cpu().numpy()
        # same cos/sin as the device: identical tap selection, values to fp32 rounding
        want = orot.rotate(img.numpy(), ang, center.numpy(), IM[interp], trig=device_trig(ang))
        assert got.shape == want.shape
        assert np.abs(got - want).max() < 1e-6, np.abs(got - want).max()
        # libm cos/sin: indices move by < 1e-4 px
        d = np.abs(got - orot.rotate(img.numpy(), ang, center.numpy(), IM[interp]))
        if interp == "nearest":
            assert (d > 0).mean() < (0.08 if case in EXACT_HALF else 0.002)
        else:
            assert d.max() < 1e-3


@pytest.mark.parametrize("case", list(ROTATE_CASES))
@pytest.mark.parametrize("interp", ["bilinear", "nearest"])
def test_fp32_matches_reference_golden(case, interp):
    z = np.load(os.path.join(GOLDEN, "rotate_ref.npz"))
    img, angle, center = make_rotate_inputs(case)
    got = bt.rotate(img.cuda(), angle.cuda()[0], center.cuda(), interp).cpu().numpy()
    d = np.abs(got - z[f"{case}_{interp}"])
    if interp == "nearest":
        assert (d > 1e-6).mean() < (0.08 if case in ("right_angle", "zero") else 0.005)
    else:
        assert d.max() < 5e-5
    assert d.mean() < 1e-4  # the reference's own acceptance metric and bound (test_rotate.py:98-102, getCost)


# the reference's own CUDA kernels, run on a B200 (tests/golden/ref_kernels_rotate.npz, make_golden_ref_kernels.py)
REFK = load_ref_kernels("rotate")


@pytest.mark.parametrize("shape,ang,ctr", [((8, 50, 50), 1.7, (25.0, 25.0)), ((7, 33, 47), 127.3, (20.5, 13.25)),
                                           ((256, 200, 200), -3.3, (100.0, 100.0)),
                                           ((32, 512, 512), 217.9, (500.0, 500.0))])  # fmt: skip
@pytest.mark.parametrize("interp", ["bilinear", "nearest"])
def test_fp32_matches_reference_cuda_kernel(shape, ang, ctr, interp):
    """Against the UNMODIFIED reference kernel: nearest must pick the same pixel everywhere (index arithmetic bit-exact,
    including the reference's FMA contraction: the whole output's digest), bilinear agrees to fp32 rounding (on a fixed,
    seeded sample of the output)."""
    g = torch.Generator().manual_seed(11)
    img = torch.randn(*shape, generator=g)
    angle, center = torch.tensor([ang]), torch.tensor(list(ctr))
    key = "fp32_" + "x".join(map(str, shape))
    check_digest(REFK, key, img, angle, center)
    got = bt.rotate(img.cuda(), angle.cuda(), center.cuda(), interp).cpu()
    if interp == "nearest":
        assert input_digest(got) == str(REFK[f"{key}_nearest"])
    else:
        got = got.numpy().reshape(-1)
        assert np.abs(got[sample_index(got.size, 2048)] - REFK[f"{key}_bilinear"]).max() < 1e-6


@pytest.mark.parametrize("case", ["bev_small", "big_angle", "off_center", "odd_c"])
@pytest.mark.parametrize("interp", ["bilinear", "nearest"])
def test_fp16_and_chw2_match_oracle(case, interp):
    img, angle, center = make_rotate_inputs(case)
    img, angle, center = img.half(), angle.half(), center.half()
    a32 = float(angle.float()[0])
    want = orot.rotate(img.float().numpy(), a32, center.float().numpy(), IM[interp], trig=device_trig(a32))
    got = bt.rotate(img.cuda(), angle.cuda(), center.cuda(), interp)
    assert got.dtype == torch.float16
    tol = 1e-3 + np.abs(want).max() * 2.0**-11
    assert np.abs(got.float().cpu().numpy() - want).max() < tol
    if interp == "nearest":  # a copy: exact
        assert np.array_equal(got.float().cpu().numpy(), want)
    # kCHW2 packed layout (RotateTRT2)
    out2 = bt.rotate_chw2(pack_chw(img[None], 2)[0].cuda(), img.shape[0], angle.cuda(), center.cuda(), interp)
    assert torch.equal(unpack_chw(out2[None].cpu(), img.shape[0])[0], got.cpu())


def test_fp16_is_closer_to_fp32_truth_than_reference_half_kernel():
    """The reference's __half kernel computes the matrix and coordinates in half precision (rotateKernel.cu:213-260);
    its own test accepts a mean-abs error of 0.5 (test_rotate.py:104-108). Ours keeps them in fp32. The reference's
    mean-abs error on these inputs was measured on a B200 (REFK)."""
    g = torch.Generator().manual_seed(3)
    img = torch.randn(16, 200, 200, generator=g)
    angle, center = torch.tensor([3.3]), torch.tensor([100.0, 100.0])
    truth = orot.rotate(img.half().float().numpy(), float(angle.half().float()[0]), center.numpy(), 0)
    ours = bt.rotate(img.half().cuda(), angle.half().cuda(), center.half().cuda(), "bilinear").float().cpu().numpy()
    check_digest(REFK, "fp16", img)
    e_ours, e_theirs = np.abs(ours - truth).mean(), float(REFK["fp16_mean_err"])
    assert e_ours < 1e-3 and e_ours <= e_theirs, (e_ours, e_theirs)


@pytest.mark.parametrize("interp", ["bilinear", "nearest"])
@pytest.mark.parametrize("half_angle", [False, True])
def test_int8_chw4_matches_dequant_oracle(interp, half_angle):
    img, angle, center = make_rotate_inputs("odd_c", seed=4)
    iq, si = quantize_per_tensor(img)
    if half_angle:
        angle, center = angle.half(), center.half()
    a32 = float(angle.float()[0])
    real = orot.rotate(iq.float().numpy() * np.float32(si), a32, center.float().numpy(), IM[interp],
                       trig=device_trig(a32))  # fmt: skip
    so = float(np.abs(real).max()) / 127.0
    out4 = bt.rotate_int8(pack_chw(iq[None], 4)[0].cuda(), si, img.shape[0], angle.cuda(), center.cuda(), so, interp)
    assert out4.dtype == torch.int8
    got = unpack_chw(out4[None].cpu(), img.shape[0])[0].float().numpy() * so
    assert np.abs(got - real).max() <= 0.5 * so + 1e-5  # one requantisation: at most half an output step


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("interp", ["bilinear", "nearest"])
def test_channels_last_entry_equals_planar(dtype, interp):
    g = torch.Generator().manual_seed(8)
    H, W, C = 50, 46, 64
    for c_odd in (8, 24, 40, 88):  # vector counts that are not a multiple of the lanes sharing a pixel
        x = torch.randn(9, 7, c_odd, generator=g).to(dtype).cuda()
        a, c = torch.tensor([-33.0]).to(dtype).cuda(), torch.tensor([3.0, 4.0]).to(dtype).cuda()
        assert torch.equal(bt.rotate_hwc(x, a, c, interp).permute(2, 0, 1),
                           bt.rotate(x.permute(2, 0, 1).contiguous(), a, c, interp))
    bev = torch.randn(H * W, 1, C, generator=g).to(dtype).cuda()  # prev_bev as BEVFormer stores it
    angle, center = torch.tensor([2.9]).to(dtype).cuda(), torch.tensor([23.0, 25.0]).to(dtype).cuda()
    planar = bt.rotate(bev.view(H, W, C).permute(2, 0, 1).contiguous(), angle, center, interp)
    hwc = bt.rotate_hwc(bev.view(H, W, C), angle, center, interp)
    assert torch.equal(hwc.permute(2, 0, 1), planar)
    # the call site's own expression (transformer.py:298-304) takes the channels-last kernel and returns a view that
    # permutes back for free
    n0 = _lib.load().b200_launch_count()
    out = bt.rotate(bev.view(H, W, C).permute(2, 0, 1), angle, center, interp)
    assert _lib.load().b200_launch_count() == n0 + 1
    assert torch.equal(out, planar)
    back = out.permute(1, 2, 0)
    assert back.is_contiguous() and torch.equal(back.reshape(H * W, 1, C), hwc.reshape(H * W, 1, C))


def test_full_size_properties():
    """BEVFormer-base prev_bev [256, 200, 200] (BASELINE configs' bev_h = bev_w = 200, embed_dims = 256)."""
    g = torch.Generator().manual_seed(1)
    img = torch.randn(256, 200, 200, generator=g).cuda()
    ctr = torch.tensor([100.0, 100.0]).cuda()
    zero, ninety = torch.tensor([0.0]).cuda(), torch.tensor([90.0]).cuda()
    assert torch.equal(bt.rotate(img, zero, ctr, "nearest"), img)
    assert (bt.rotate(img, zero, ctr, "bilinear") - img).abs().max().item() < 1e-3  # index rounding x gradient
    assert torch.equal(bt.rotate(img, ninety, ctr, "nearest"), torch.rot90(img, 1, (1, 2)))
    a = torch.tensor([7.3]).cuda()
    other = torch.randn(256, 200, 200, generator=g).cuda()
    lin = bt.rotate(img + 2 * other, a, ctr, "bilinear")
    assert (lin - (bt.rotate(img, a, ctr, "bilinear") + 2 * bt.rotate(other, a, ctr, "bilinear"))).abs().max() < 1e-4
    # a full turn more is the same rotation up to fp32 rounding of the angle
    again = bt.rotate(img, a + 360.0, ctr, "bilinear")
    assert (again - bt.rotate(img, a, ctr, "bilinear")).abs().max().item() < 1e-2
    # pixels whose pre-image is outside the image are zero: rotating an all-ones image keeps values in [0, 1]
    ones = bt.rotate(torch.ones(4, 200, 200).cuda(), torch.tensor([45.0]).cuda(), ctr, "bilinear")
    assert ones.min().item() >= 0.0 and ones.max().item() <= 1.0 + 1e-6 and ones[:, 0, 0].abs().max().item() == 0.0


def test_errors_and_edge_cases():
    img = torch.randn(4, 9, 11)
    with pytest.raises(RuntimeError):
        bt.rotate(img, torch.tensor(1.0), torch.tensor([4.0, 4.0]))  # CPU tensor: no fallback
    with pytest.raises(RuntimeError):
        bt.rotate(img[None].cuda(), torch.tensor(1.0), torch.tensor([4.0, 4.0]))  # ndim != 3 (rotate.py:14)
    with pytest.raises(ValueError):
        bt.rotate(img.cuda(), torch.tensor([1.0, 2.0]), torch.tensor([4.0, 4.0]))
    with pytest.raises(KeyError):
        bt.rotate(img.cuda(), torch.tensor(1.0), torch.tensor([4.0, 4.0]), "bicubic")  # _MODE lookup, as the reference
    with pytest.raises(_lib.B200OpsError):
        bt.rotate(img.double().cuda(), torch.tensor(1.0), torch.tensor([4.0, 4.0]))
    with pytest.raises(_lib.B200OpsError):  # channels-last needs C % 4 == 0
        bt.rotate_hwc(torch.randn(9, 11, 6).cuda(), torch.tensor(1.0), torch.tensor([4.0, 4.0]))
    lib = _lib.load()
    x = img.cuda()
    a, c = torch.tensor([1.0]).cuda(), torch.tensor([4.0, 4.0]).cuda()
    dims = (ctypes.c_int * 3)(4, 9, 11)
    assert lib.b200_rotate_f32(x.data_ptr(), x.data_ptr(), a.data_ptr(), c.data_ptr(), dims, 2, None) == 2
    assert lib.b200_rotate_f32(None, x.data_ptr(), a.data_ptr(), c.data_ptr(), dims, 0, None) == 2
    assert lib.b200_rotate_f32(x.data_ptr(), x.data_ptr(), a.data_ptr(), c.data_ptr(), (ctypes.c_int * 3)(4, 0, 11), 0,
                               None) == 2  # fmt: skip
    # non-finite angle: every source index is replaced by -100 (safe_downgrade_to_int_range) -> all zeros, no fault
    out = bt.rotate(x, torch.tensor([float("inf")]).cuda(), c, "bilinear")
    assert torch.equal(out, torch.zeros_like(out))
    # 1x1 image, python-number angle / tuple centre
    one = bt.rotate(torch.ones(3, 1, 1).cuda(), 0.0, (0.5, 0.5), "bilinear")
    assert torch.allclose(one, torch.ones(3, 1, 1).cuda())


def test_same_box_timing_against_reference_kernel():
    """At BEVFormer-base size, device time per call (CUDA events around 20 back-to-back launches) of this library against
    the reference's rotateKernel<float|__half>, timed the same way on a B200 (REFK: the best of 5 such runs; the card and
    its power limit are stored with the numbers)."""

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
    res = {}
    for tag, x, a, c in (("f32", img, angle, center), ("f16", img.half(), angle.half(), center.half())):
        res[f"reference_{tag}_us"] = float(REFK[f"time_reference_{tag}_us"])
        res[f"b200_{tag}_us"] = timed(lambda: bt.rotate(x, a, c, "bilinear"))
        hwc = x.permute(1, 2, 0).contiguous()
        res[f"b200_hwc_{tag}_us"] = timed(lambda: bt.rotate_hwc(hwc, a, c, "bilinear"))
    print(f"\n[rotate timing] {res} (reference on {REFK['time_device']})")
    assert res["b200_f32_us"] < res["reference_f32_us"] and res["b200_f16_us"] < res["reference_f16_us"], res
