"""GPU parity tests for DCNv2 (pytest -m gpu). Checkers: oracle/dcn (reference im2col restated + fp64-accumulated GEMM),
torchvision.ops.deform_conv2d on the GPU at larger sizes, and the reference's own CUDA launcher run on a B200.
Tolerances: FP32 1e-4 relative to max|out| (GEMM summation order). FP16, against the FP32 formulas evaluated on the
FP16-rounded inputs: half an FP16 spacing of the largest |out| (the output rounding no FP16-out kernel can avoid; 1.95e-3
for |out| in [4, 8)) + north_star's 1e-3 for everything before it (`fp16_tol`; measured 1e-4..2e-4 of the 1e-3 are used).
The reference's own FP16 bar is mean-abs 0.05 (test_modulated_deformable_conv2d.py:100-103)."""
import numpy as np
import pytest
import torch

import bevformer_tensorrt_b200 as bt


def fp16_tol(want):
    """FP16-output error budget: 0.5 * spacing_fp16(max|want|) + 1e-3 (see the module docstring)."""
    return 0.5 * float(np.spacing(np.float16(np.abs(want).max()))) + 1e-3
from bevformer_tensorrt_b200 import _lib
from oracle import dcn as odcn
from tests.helpers import DCN_CASES, check_digest, load_ref_kernels, make_dcn_inputs, sample_index

pytestmark = pytest.mark.gpu


def _call(fn, x, off, mask, w, b, kw):
    return fn(x.cuda(), off.cuda(), mask.cuda(), w.cuda(), b.cuda() if b is not None else None, kw["stride"],
              kw["padding"], kw["dilation"], kw["groups"], kw["deform_groups"])  # fmt: skip


@pytest.mark.parametrize("case", list(DCN_CASES))
def test_fp32_matches_oracle(case):
    x, off, mask, w, b, kw = make_dcn_inputs(case)
    want = odcn.modulated_deformable_conv2d(x.numpy(), off.numpy(), mask.numpy(), w.numpy(), b.numpy(), **kw)
    for fn in (bt.modulated_deformable_conv2d, bt.modulated_deformable_conv2d2):
        got = _call(fn, x, off, mask, w, b, kw).cpu().numpy()
        assert got.shape == want.shape
        assert np.abs(got - want).max() < 1e-4 * max(1.0, np.abs(want).max()), (case, np.abs(got - want).max())
    nb = _call(bt.modulated_deformable_conv2d, x, off, mask, w, None, kw).cpu().numpy()  # bias optional (4 inputs)
    assert np.abs(nb - (want - b.numpy()[None, :, None, None])).max() < 2e-4 * max(1.0, np.abs(want).max())


FUSED_CASES = ["fused_co128", "fused_co256_ragged", "fused_co512_s2", "fused_k1"]


@pytest.mark.parametrize("case", FUSED_CASES)
def test_fp16_fused_tcgen05_path_matches_oracle_and_gather_gemm_path(case):
    """The fused implicit-GEMM kernel (csrc/dcn_fused.cu) against the oracle and against the library's own generic
    hand-written kernel (csrc/dcn_generic.cu) on the same inputs."""
    x, off, mask, w, b, kw = make_dcn_inputs(case, dtype=torch.float16)
    want = odcn.modulated_deformable_conv2d(*(t.float().numpy() for t in (x, off, mask, w, b)), **kw)
    lib = _lib.load()
    prev = lib.b200_dcn_set_fused(1)
    try:
        fused = _call(bt.modulated_deformable_conv2d, x, off, mask, w, b, kw)
        lib.b200_dcn_set_fused(0)
        plain = _call(bt.modulated_deformable_conv2d, x, off, mask, w, b, kw)
    finally:
        lib.b200_dcn_set_fused(prev)
    # Error budget (FP16 in, FP16 out, FP32 accumulation over K = kh*kw*C): (1) the FP16 rounding of the OUTPUT, half a
    # spacing of the largest |out| — unavoidable, 1.95e-3 at |out| in [4, 8) — plus (2) everything before it: FP16
    # columns (the reference's im2col buffer is FP16 too, …Conv2dKernel.cu:321-388) and the packed-HFMA2 corner blend,
    # both 2^-11 relative per term and averaged over K >= 576 terms, measured 1e-4 .. 2e-4; north_star's 1e-3 covers (2).
    tol = fp16_tol(want)
    print(f"[dcn fp16 {case}] max|want| {np.abs(want).max():.3f}  err fused {np.abs(fused.float().cpu().numpy() - want).max():.2e}"
          f"  err generic {np.abs(plain.float().cpu().numpy() - want).max():.2e}  fp16 spacing at max "
          f"{np.spacing(np.float16(np.abs(want).max())):.2e}")
    assert np.abs(fused.float().cpu().numpy() - want).max() < tol, np.abs(fused.float().cpu().numpy() - want).max()
    assert np.abs(plain.float().cpu().numpy() - want).max() < tol
    nb = _call(bt.modulated_deformable_conv2d, x, off, mask, w, None, kw)  # no bias
    assert np.abs(nb.float().cpu().numpy() - (want - b.float().numpy()[None, :, None, None])).max() < tol


def test_fp16_fused_channels_last_input_and_packed_weight_cache():
    x, off, mask, w, b, kw = make_dcn_inputs("fused_co256_ragged", dtype=torch.float16)
    args = [t.cuda() for t in (x, off, mask, w, b)]
    want = bt.modulated_deformable_conv2d(*args, kw["stride"], kw["padding"], kw["dilation"], 1, 1)
    x_cl = args[0].contiguous(memory_format=torch.channels_last)  # NHWC bytes: consumed without the transpose pre-pass
    got = bt.modulated_deformable_conv2d(x_cl, *args[1:], kw["stride"], kw["padding"], kw["dilation"], 1, 1)
    assert torch.equal(got, want)
    again = bt.modulated_deformable_conv2d(*args, kw["stride"], kw["padding"], kw["dilation"], 1, 1)  # cached weights
    assert torch.equal(again, want)
    args[3].mul_(2.0)  # in-place weight update bumps the version: the cache must not serve stale weights
    upd = bt.modulated_deformable_conv2d(*args, kw["stride"], kw["padding"], kw["dilation"], 1, 1)
    assert not torch.equal(upd, want)


def test_packed_weight_cache_is_tied_to_the_weight_object():
    """ADVICE r1: the packed-weight cache must never serve another tensor's weights. Entries live and die with the
    nn.Parameter they were packed from; temporaries are packed per call."""
    import gc

    import importlib

    mod = importlib.import_module("bevformer_tensorrt_b200.functions.modulated_deformable_conv2d")

    x, off, mask, w, b, kw = make_dcn_inputs("fused_co128", dtype=torch.float16)
    xs = [t.cuda() for t in (x, off, mask)]
    call = lambda wt: bt.modulated_deformable_conv2d(*xs, wt, b.cuda(), kw["stride"], kw["padding"], kw["dilation"], 1, 1)  # noqa: E731
    p1 = torch.nn.Parameter(w.cuda(), requires_grad=False)
    n0 = len(mod._PACKED)
    out1 = call(p1)
    assert len(mod._PACKED) == n0 + 1
    l0 = _lib.launch_count()
    assert torch.equal(call(p1), out1)
    cached_launches = _lib.launch_count() - l0
    l0 = _lib.launch_count()
    assert torch.equal(call(w.cuda()), out1)  # a temporary: same values, packed on the spot, never cached
    assert _lib.launch_count() - l0 == cached_launches + 1 and len(mod._PACKED) == n0 + 1
    del p1
    gc.collect()
    assert len(mod._PACKED) == n0  # the entry died with its weight
    p2 = torch.nn.Parameter((w * 3).cuda(), requires_grad=False)  # same shape, very likely the same address
    out2 = call(p2)
    assert torch.equal(out2, call((w * 3).cuda())) and not torch.equal(out2, out1)


@pytest.mark.parametrize("case", ["k3_s1_p1_g2_dg2", "fused_co128", "k3x5_s1_p1_g1_dg1"])
def test_fp16_chw2_entry_equals_linear_entry(case):
    """kCHW2 packets (…TRT2 format table, …Conv2dPlugin.cpp:222-250) in, the same bits out as the linear FP16 entry."""
    from bevformer_tensorrt_b200.functions.grid_sampler import pack_chw
    from bevformer_tensorrt_b200.functions.modulated_deformable_conv2d import modulated_deformable_conv2d_chw2

    x, off, mask, w, b, kw = make_dcn_inputs(case, dtype=torch.float16)
    want = _call(bt.modulated_deformable_conv2d, x, off, mask, w, b, kw)
    got = modulated_deformable_conv2d_chw2(pack_chw(x, 2).cuda(), pack_chw(off, 2).cuda(), mask.cuda(), pack_chw(w, 2).cuda(),
                                           b.cuda(), x.shape[1], kw["stride"], kw["padding"], kw["dilation"], kw["groups"],
                                           kw["deform_groups"])  # fmt: skip
    assert torch.equal(got, want)


def test_dcnv2p_layer_runs_the_plugin_op():
    """DCNv2P / DCNv2P2 (det2trt/models/modules/cnn/dcn.py:31-164) at the reference op test's structure: groups = 2,
    deform_groups = 2 (test_modulated_deformable_conv2d.py:6-11,37): conv_offset -> (offset, sigmoid(mask)) -> op."""
    from bevformer_tensorrt_b200.modules import CONV_LAYERS

    torch.manual_seed(0)
    for name, dt in (("DCNv2P", torch.float32), ("DCNv2P2", torch.float16)):
        layer = CONV_LAYERS[name](16, 12, 3, stride=1, padding=1, groups=2, deform_groups=2).cuda()
        layer.conv_offset.weight.data.normal_(0, 0.05)
        layer.conv_offset.bias.data.normal_(0, 0.5)
        layer.bias.data.normal_()
        layer = layer.to(dt)
        x = torch.randn(2, 16, 13, 17, device="cuda", dtype=dt)
        got = layer(x)
        o = layer.conv_offset(x)
        o1, o2, m = torch.chunk(o, 3, dim=1)
        npf = lambda t_: t_.detach().float().cpu().numpy()  # noqa: E731
        want = odcn.modulated_deformable_conv2d(npf(x), npf(torch.cat((o1, o2), 1)), npf(torch.sigmoid(m)),
                                                npf(layer.weight), npf(layer.bias), stride=1, padding=1, dilation=1,
                                                groups=2, deform_groups=2)  # fmt: skip
        assert got.shape == (2, 12, 13, 17) and got.dtype == dt
        tol = 1e-4 if dt == torch.float32 else 5e-3
        assert np.abs(npf(got) - want).max() < tol * max(1.0, np.abs(want).max())


@pytest.mark.parametrize("case", ["k3_s1_p1_g2_dg2", "backbone_like", "k3_s2_p1_g1_dg1"])
def test_fp16_matches_oracle(case):
    x, off, mask, w, b, kw = make_dcn_inputs(case, dtype=torch.float16)
    want = odcn.modulated_deformable_conv2d(*(t.float().numpy() for t in (x, off, mask, w, b)), **kw)
    got = _call(bt.modulated_deformable_conv2d, x, off, mask, w, b, kw)
    assert got.dtype == torch.float16
    err = np.abs(got.float().cpu().numpy() - want).max()
    assert err < fp16_tol(want), (case, err, fp16_tol(want))


def test_im2col_indices_bit_exact_through_identity_weights():
    """With a 1x1 kernel, identity weights and mask 1 the op returns the bilinear sample itself; integer-valued offsets
    then return exact pixels of an index image, so the device's h_im/w_im/floor arithmetic is compared bit-exactly."""
    C, H, W = 4, 19, 23
    img = torch.arange(H * W, dtype=torch.float32).view(1, 1, H, W).repeat(1, C, 1, 1) + 1.0
    g = torch.Generator().manual_seed(5)
    off = torch.randint(-6, 7, (1, 2, H, W), generator=g).float()
    mask = torch.ones(1, 1, H, W)
    w = torch.eye(C).view(C, C, 1, 1)
    want = odcn.modulated_deformable_conv2d(img.numpy(), off.numpy(), mask.numpy(), w.numpy(), None)
    got = bt.modulated_deformable_conv2d(img.cuda(), off.cuda(), mask.cuda(), w.cuda(), None).cpu().numpy()
    assert np.array_equal(got, want)


def test_base_backbone_shape_against_torchvision_gpu():
    """BEVFormer-base R101 stage-3 DCN shape [6,256,58,100] 3x3 (SURVEY §8a a13), FP32, vs torchvision on the same GPU."""
    import torchvision

    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(6, 256, 58, 100, device="cuda", generator=g)
    off = torch.randn(6, 18, 58, 100, device="cuda", generator=g) * 2
    mask = torch.sigmoid(torch.randn(6, 9, 58, 100, device="cuda", generator=g))
    w = torch.randn(256, 256, 3, 3, device="cuda", generator=g) / 48.0
    b = torch.randn(256, device="cuda", generator=g)
    want = torchvision.ops.deform_conv2d(x, off, w, b, padding=1, mask=mask)
    got = bt.modulated_deformable_conv2d(x, off, mask, w, b, 1, 1, 1, 1, 1)
    assert (got - want).abs().max().item() < 2e-3  # both sides may use TF32-free fp32 GEMMs with different orders
    # FP16 op (the fused tcgen05 kernel at this shape) against the same FP32 formulas on the FP16-rounded inputs
    h = [t.half() for t in (x, off, mask, w, b)]
    want16 = torchvision.ops.deform_conv2d(h[0].float(), h[1].float(), h[3].float(), h[4].float(), padding=1, mask=h[2].float())
    goth = bt.modulated_deformable_conv2d(h[0], h[1], h[2], h[3], h[4], 1, 1, 1, 1, 1)
    err16 = (goth.float() - want16).abs().max().item()
    print(f"[dcn fp16 base layer] max|want| {want16.abs().max().item():.3f} err {err16:.2e} budget {fp16_tol(want16.cpu().numpy()):.2e}")
    assert err16 < fp16_tol(want16.cpu().numpy())


@pytest.mark.parametrize("case", ["k3_s1_p1_g2_dg2", "backbone_like"])
def test_fp32_matches_reference_launcher(case):
    """Against the reference's own CUDA launcher run on a B200 (tests/golden/ref_kernels_dcn.npz, on a fixed, seeded
    sample of the output elements; make_golden_ref_kernels.py)."""
    z = load_ref_kernels("dcn")
    x, off, mask, w, b, kw = make_dcn_inputs(case)
    check_digest(z, f"fp32_{case}", x, off, mask, w, b)
    got = _call(bt.modulated_deformable_conv2d, x, off, mask, w, b, kw).cpu().numpy().reshape(-1)
    want = z[f"fp32_{case}"]
    assert np.abs(got[sample_index(got.size, 2048)] - want).max() < 1e-4 * max(1.0, float(z[f"fp32_{case}_amax"]))


def test_error_behaviour():
    x, off, mask, w, b, kw = make_dcn_inputs("k3_s2_p1_g1_dg1")
    with pytest.raises(RuntimeError):
        bt.modulated_deformable_conv2d(x, off, mask, w, b, 2, 1, 1, 1, 1)
    with pytest.raises(ValueError):
        bt.modulated_deformable_conv2d(x.cuda(), off.cuda()[:, :-1], mask.cuda(), w.cuda(), b.cuda(), 2, 1, 1, 1, 1)
    lib = _lib.load()
    # channels not divisible by groups: the reference exit(1)s, here status 1
    assert lib.b200_dcn_f32(1, 1, None, 1, 1, 1, 1, 1, 6, 4, 4, 4, 3, 3, 1, 1, 1, 1, 1, 1, 4, 1, 1, None, None) == 1
    assert lib.b200_dcn_f32(None, None, None, None, None, None, None, 1, 4, 4, 4, 4, 3, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1,
                            None, None) == 2


@pytest.mark.parametrize("bias_dtype", [torch.float32, torch.float16, None])
@pytest.mark.parametrize("case", ["fused_co128", "fused_co256_ragged", "fused_co512_s2"])
def test_int8_matches_dequant_oracle(case, bias_dtype):
    """INT8 DCN: int8 kCHW4 input / weight, int8 offset / mask, per-tensor MinMax scales; checked against the FP32
    formulas on the dequantised tensors, requantised with T2int8. Tolerance: the FP16 rounding of the sampled columns
    (2^-11 relative on values <= 127 in input-scale units) summed over K, expressed in output steps."""
    from bevformer_tensorrt_b200.functions.grid_sampler import pack_chw
    from bevformer_tensorrt_b200.workloads import quantize_per_tensor

    x, off, mask, w, b, kw = make_dcn_inputs(case)
    xq, si = quantize_per_tensor(x)
    oq, so_ = quantize_per_tensor(off)
    mq, sm = quantize_per_tensor(mask)
    wq, sw = quantize_per_tensor(w)
    bias = None if bias_dtype is None else b.to(bias_dtype)
    real = odcn.modulated_deformable_conv2d(xq.float().numpy() * si, oq.float().numpy() * so_, mq.float().numpy() * sm,
                                            wq.float().numpy() * sw, None if bias is None else bias.float().numpy(), **kw)
    sout = float(np.abs(real).max()) / 127.0
    got = bt.modulated_deformable_conv2d_int8(
        pack_chw(xq, 4).cuda(), si, oq.cuda(), so_, mq.cuda(), sm, pack_chw(wq, 4).cuda(), sw,
        None if bias is None else bias.cuda(), sout, x.shape[1], kw["stride"], kw["padding"], kw["dilation"], 1, 1)
    assert got.dtype == torch.int8 and tuple(got.shape) == real.shape
    err = np.abs(got.cpu().numpy().astype(np.float32) * sout - real).max()
    assert err <= 0.75 * sout, (err, sout)  # half a step from the requantisation + fp16 column rounding
    # tensors that do not match the declared deform_groups are rejected before anything is launched
    with pytest.raises(ValueError):
        bt.modulated_deformable_conv2d_int8(pack_chw(xq, 4).cuda(), si, oq.cuda(), so_, mq.cuda(), sm,
                                            pack_chw(wq, 4).cuda(), sw, None, sout, x.shape[1], kw["stride"],
                                            kw["padding"], kw["dilation"], 1, 2)


@pytest.mark.parametrize("case", ["k3_s1_p1_g2_dg2", "k3_s2_p1_g1_dg1", "k3_s1_p2_d2_g1_dg4", "k3x5_s1_p1_g1_dg1",
                                  "backbone_like"])  # fmt: skip
def test_int8_unfused_shapes_match_dequant_oracle(case):
    """INT8 for the shapes the fused kernel does not take (groups / deformable groups > 1, small or odd channel
    counts): dequantise -> generic hand-written FP16 kernel -> one requantisation."""
    from bevformer_tensorrt_b200.functions.grid_sampler import pack_chw
    from bevformer_tensorrt_b200.workloads import quantize_per_tensor

    x, off, mask, w, b, kw = make_dcn_inputs(case)
    xq, si = quantize_per_tensor(x)
    oq, so_ = quantize_per_tensor(off)
    mq, sm = quantize_per_tensor(mask)
    wq, sw = quantize_per_tensor(w)
    real = odcn.modulated_deformable_conv2d(xq.float().numpy() * si, oq.float().numpy() * so_, mq.float().numpy() * sm,
                                            wq.float().numpy() * sw, b.numpy(), **kw)
    sout = float(np.abs(real).max()) / 127.0
    got = bt.modulated_deformable_conv2d_int8(
        pack_chw(xq, 4).cuda(), si, oq.cuda(), so_, mq.cuda(), sm, pack_chw(wq, 4).cuda(), sw, b.cuda(), sout,
        x.shape[1], kw["stride"], kw["padding"], kw["dilation"], kw["groups"], kw["deform_groups"])
    assert got.dtype == torch.int8 and tuple(got.shape) == real.shape
    err = np.abs(got.cpu().numpy().astype(np.float32) * sout - real).max()
    assert err <= 0.75 * sout, (err, sout)
