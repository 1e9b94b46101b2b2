"""GPU tests of the plugin-shaped C entries b200_grid_sampler_enqueue and b200_dcn_enqueue (csrc/api.cu) — the code a
TensorRT engine runs through csrc/trt_plugin/b200_trt_plugins.cpp — and of DCN at non-square kernels with asymmetric
stride / padding / dilation on an H != W input, where an h/w swap anywhere on the DCN path shows.

Descriptors are built the way TensorRT hands them over: b200_tensor_desc with the logical (unpacked) NCHW dims, type
0 f32 / 1 f16 / 2 i8 / 3 i32, format 0 linear / 1 kCHW2 / 3 kCHW4, per-tensor scales for INT8. Every enqueue output is
compared bit for bit with the Python op that reaches the same launcher, and with the oracle:
  * grid sampler: oracle/grid_sampler.py (2-D: the reference kernel's formulas in C; 3-D: the reference binding's
    aten.grid_sampler evaluated in float64). FP32 1e-5, FP16 1e-3 + max|want| * 2^-11, INT8 half an output step on the
    dequantised tensors. Nearest mode is checked through the sampled index, never through a value tolerance.
  * DCN: oracle/dcn.py (fp64-accumulated GEMM) with the budgets of tests/test_dcn_gpu.py: FP32 1e-4 * max(1, max|want|),
    FP16 `fp16_tol`, INT8 0.75 output steps.
Outputs and the DCN workspace are the front of larger buffers whose tail holds a known byte pattern, so an entry that
writes past the size it asked for fails a test instead of corrupting memory."""
import ctypes
import functools
import importlib
import itertools

import numpy as np
import pytest
import torch

import bevformer_tensorrt_b200 as bt
from bevformer_tensorrt_b200 import _lib
from bevformer_tensorrt_b200.functions.grid_sampler import pack_chw, unpack_chw
from bevformer_tensorrt_b200.functions.modulated_deformable_conv2d import (modulated_deformable_conv2d_chw2,
                                                                          modulated_deformable_conv2d_int8)
from bevformer_tensorrt_b200.workloads import quantize_per_tensor
from oracle import dcn as odcn
from oracle import grid_sampler as ogs
from tests.helpers import DCN_CASES, make_dcn_inputs, make_grid_sampler_inputs
from tests.test_dcn_gpu import fp16_tol

pytestmark = pytest.mark.gpu

F32, F16, I8, I32 = 0, 1, 2, 3  # nvinfer1::DataType
LINEAR, CHW2, CHW4 = 0, 1, 3  # nvinfer1::TensorFormat
OK, UNSUPPORTED, BAD_PARAM = 0, 1, 2
GUARD, PATTERN = 4096, 0xA5


def desc(shape, ttype, fmt=LINEAR, scale=1.0):
    d = _lib.TensorDesc()
    d.dims.nbDims = len(shape)
    for i, s in enumerate(shape):
        d.dims.d[i] = int(s)
    d.type, d.format, d.scale = ttype, fmt, float(scale)
    return d


def descs(*ds):
    return (_lib.TensorDesc * len(ds))(*ds)


def ptrs(*ts):
    return (ctypes.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


def ints(*v):
    return (ctypes.c_int * len(v))(*v)


class Guarded:
    """A tensor of `shape` at the front of a byte buffer with GUARD bytes of PATTERN behind it."""

    def __init__(self, shape, dtype, nbytes=None):
        self.nbytes = int(np.prod(shape)) * torch.empty(0, dtype=dtype).element_size() if nbytes is None else nbytes
        self.buf = torch.full((self.nbytes + GUARD,), PATTERN, dtype=torch.uint8, device="cuda")
        self.t = self.buf[: int(np.prod(shape)) * torch.empty(0, dtype=dtype).element_size()].view(dtype).view(shape)

    def intact(self):
        return bool((self.buf[self.nbytes:] == PATTERN).all())


# ---------------------------------------------------------------------------------------------------------------------
# Grid sampler
MODES = list(itertools.product(["bilinear", "nearest", "bicubic"], ["zeros", "border", "reflection"], [False, True]))
IM = {"bilinear": 0, "nearest": 1, "bicubic": 2}
PM = {"zeros": 0, "border": 1, "reflection": 2}
GS_FORMS = ["f32", "f16", "f16_chw2", "i8_chw4"]
GS_SHAPE = (2, 37, 11, 13, 21, 27)  # N, C (odd: partial kCHW2 / kCHW4 packets), Hi, Wi, Ho, Wo (partial tiles)


def _gs_enqueue(io, inputs, out, mode, use_h2=0):
    """Asserts supportsFormatCombination accepts every position of `io`, then runs the enqueue."""
    lib = _lib.load()
    for pos in range(3):
        assert lib.b200_grid_sampler_supports_format(pos, descs(*io), 2, 1, use_h2) == 1, pos
    interp, pad, align = mode
    st = lib.b200_grid_sampler_enqueue(descs(*io[:2]), descs(io[2]), ptrs(*inputs), ptrs(out), None,
                                       _lib.current_stream_ptr(), IM[interp], PM[pad], int(align))  # fmt: skip
    torch.cuda.synchronize()
    return st


@pytest.mark.parametrize("form", GS_FORMS)
@pytest.mark.parametrize("interp,pad,align", MODES)
def test_grid_sampler_2d_enqueue_matches_python_op_and_oracle(interp, pad, align, form):
    N, C, Hi, Wi, Ho, Wo = GS_SHAPE
    mode = (interp, pad, align)
    inp, grid = make_grid_sampler_inputs(N, C, Hi, Wi, Ho, Wo, seed=41)
    ind, gdd, odd = (N, C, Hi, Wi), (N, 2, Ho, Wo), (N, C, Ho, Wo)
    if form in ("f32", "f16"):
        dt, tt = (torch.float32, F32) if form == "f32" else (torch.float16, F16)
        x, g = inp.to(dt).cuda(), grid.to(dt).cuda()
        out = Guarded(odd, dt)
        assert _gs_enqueue([desc(ind, tt), desc(gdd, tt), desc(odd, tt)], [x, g], out.t, mode) == OK
        assert torch.equal(out.t, bt.grid_sampler(x, g, interp, pad, align))
        got = out.t.float().cpu().numpy()
        want = ogs.grid_sample_2d(x.float().cpu().numpy(), g.float().cpu().numpy(), IM[interp], PM[pad], align)
        tol = 1e-5 if form == "f32" else 1e-3 + np.abs(want).max() * 2.0**-11
    elif form == "f16_chw2":
        xh, gh = inp.half(), grid.half()
        x2, g2 = pack_chw(xh, 2).cuda(), pack_chw(gh, 2).cuda()  # grid: [N, 1, Ho, Wo, 2] = (x, y)
        out = Guarded((N, (C + 1) // 2, Ho, Wo, 2), torch.float16)
        io = [desc(ind, F16, CHW2), desc(gdd, F16, CHW2), desc(odd, F16, CHW2)]
        assert _gs_enqueue(io, [x2, g2], out.t, mode, use_h2=1) == OK
        got = unpack_chw(out.t.cpu(), C)
        assert torch.equal(got, unpack_chw(bt.grid_sampler_chw2(x2, g2, C, interp, pad, align).cpu(), C))
        got = got.float().numpy()
        want = ogs.grid_sample_2d(xh.float().numpy(), gh.float().numpy(), IM[interp], PM[pad], align)
        tol = 1e-3 + np.abs(want).max() * 2.0**-11
    else:
        iq, si = quantize_per_tensor(inp)
        gq, sg = quantize_per_tensor(grid)
        want = ogs.grid_sample_2d(iq.float().numpy() * si, gq.float().numpy() * sg, IM[interp], PM[pad], align)
        so = float(np.abs(want).max()) / 127.0
        x4, g4 = pack_chw(iq, 4).cuda(), pack_chw(gq, 4).cuda()  # grid: [N, 1, Ho, Wo, 4] = (x, y, 0, 0)
        out = Guarded((N, (C + 3) // 4, Ho, Wo, 4), torch.int8)
        io = [desc(ind, I8, CHW4, si), desc(gdd, I8, CHW4, sg), desc(odd, I8, CHW4, so)]
        assert _gs_enqueue(io, [x4, g4], out.t, mode) == OK
        got = unpack_chw(out.t.cpu(), C)
        py = bt.grid_sampler_int8(x4, si, g4, sg, so, C, interp, pad, align)
        assert torch.equal(got, unpack_chw(py.cpu(), C))
        got = got.float().numpy() * so
        tol = 0.5 * so + 1e-6  # one requantisation
    assert out.intact()
    err = np.abs(got - want).max()
    assert err <= tol, (form, mode, err, tol)


def _index_grid_3d(N, sizes_dhw, out_dhw, align, seed):
    """A [-10, 10] grid [N, 3, Do, Ho, Wo] whose source coordinates are integer + u, |u| <= 0.4, from two pixels
    before the image to two after it: nearest rounding is never near a tie, also after reflection or fp16 rounding of
    the grid, so the sampled index is defined exactly."""
    g = torch.Generator().manual_seed(seed)
    planes = []
    for size in reversed(sizes_dhw):  # x (W), y (H), z (D)
        k = torch.randint(-2, size + 2, (N, *out_dhw), generator=g).double()
        c = k + (torch.rand((N, *out_dhw), generator=g, dtype=torch.float64) - 0.5) * 0.8
        planes.append(10 * (2 * c / (size - 1) - 1) if align else 10 * ((2 * c + 1) / size - 1))
    return torch.stack(planes, 1).float()


@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("pad", ["zeros", "border", "reflection"])
@pytest.mark.parametrize("interp", ["bilinear", "nearest"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_grid_sampler_3d_enqueue_matches_python_op_and_float64_binding(dtype, interp, pad, align):
    """5-D through the enqueue: bilinear against the reference binding's aten.grid_sampler in float64 on the same
    (fp16-rounded) tensors; nearest on an image whose value is its own flat index (+1, distinct per batch and channel,
    all exact in fp16), compared exactly."""
    N, C, (Di, Hi, Wi), (Do, Ho, Wo) = 2, 5, (4, 6, 7), (5, 7, 9)
    if interp == "bilinear":
        inp, grid = make_grid_sampler_inputs(N, C, Hi, Wi, Ho, Wo, seed=43, depth=(Di, Do))
    else:
        inp = torch.arange(1, N * C * Di * Hi * Wi + 1, dtype=torch.float32).view(N, C, Di, Hi, Wi)
        grid = _index_grid_3d(N, (Di, Hi, Wi), (Do, Ho, Wo), align, seed=44)
    x, g = inp.to(dtype).cuda(), grid.to(dtype).cuda()
    tt = F32 if dtype == torch.float32 else F16
    ind, gdd, odd = (N, C, Di, Hi, Wi), (N, 3, Do, Ho, Wo), (N, C, Do, Ho, Wo)
    out = Guarded(odd, dtype)
    assert _gs_enqueue([desc(ind, tt), desc(gdd, tt), desc(odd, tt)], [x, g], out.t, (interp, pad, align)) == OK
    assert out.intact()
    assert torch.equal(out.t, bt.grid_sampler(x, g, interp, pad, align))
    want = ogs.grid_sampler_torch_port(x.cpu().double(), g.cpu().double(), IM[interp], PM[pad], align).numpy()
    got = out.t.cpu().double().numpy()
    if interp == "nearest":
        assert np.array_equal(got, want), (pad, align, int((got != want).sum()))
        assert np.unique(want).size > 100  # the grid really walks over the image
        return
    # FP32: the kernel unnormalises in fp32 (a few 1e-6 px) times the neighbour differences of an N(0, 1) image
    tol = 3e-5 if dtype == torch.float32 else 1e-3 + np.abs(want).max() * 2.0**-11
    assert np.abs(got - want).max() <= tol, (pad, align, np.abs(got - want).max())


def test_grid_sampler_enqueue_unsupported_forms_launch_nothing():
    """5-D int8, 5-D kCHW2 and 5-D bicubic (the reference's plugin has none of them) and an unknown dtype: status 1."""
    lib = _lib.load()
    N, C, (Di, Hi, Wi), (Do, Ho, Wo) = 1, 4, (3, 4, 5), (2, 3, 4)
    x = torch.zeros(N * C * Di * Hi * Wi * 4, dtype=torch.uint8, device="cuda")
    g = torch.zeros(N * 3 * Do * Ho * Wo * 4, dtype=torch.uint8, device="cuda")
    out = Guarded((N * C * Do * Ho * Wo * 4,), torch.uint8)
    ind, gdd, odd = (N, C, Di, Hi, Wi), (N, 3, Do, Ho, Wo), (N, C, Do, Ho, Wo)
    cases = [(I8, CHW4, 0), (F16, CHW2, 0), (F32, LINEAR, 2), (F16, LINEAR, 2), (I32, LINEAR, 0)]
    for (tt, fmt, interp), dims in itertools.product(cases, [(ind, gdd, odd), ((N, C, Hi, Wi), (N, 2, Ho, Wo),
                                                                               (N, C, Ho, Wo))]):  # fmt: skip
        if len(dims[0]) == 4 and tt != I32:
            continue  # 4-D: only the unknown dtype
        l0 = lib.b200_launch_count()
        st = lib.b200_grid_sampler_enqueue(descs(desc(dims[0], tt, fmt), desc(dims[1], tt, fmt)),
                                           descs(desc(dims[2], tt, fmt)), ptrs(x, g), ptrs(out.t), None,
                                           _lib.current_stream_ptr(), interp, 0, 0)  # fmt: skip
        assert st == UNSUPPORTED, (tt, fmt, interp, len(dims[0]), st)
        assert lib.b200_launch_count() == l0
    torch.cuda.synchronize()
    assert out.intact() and bool((out.t == PATTERN).all())


def test_grid_sampler_enqueue_rejects_an_output_that_disagrees_with_input_and_grid():
    """The launcher takes N and C from the input and the output extent from the grid. An output descriptor that says
    otherwise would be written past its end: status 2, nothing launched. Every buffer here is sized for the largest
    geometry in play, so no call can touch memory it does not own."""
    lib = _lib.load()
    N, C, Hi, Wi, Ho, Wo = 2, 6, 9, 10, 7, 8
    inp, grid = make_grid_sampler_inputs(N, C, Hi, Wi, Ho, Wo, seed=45)
    x, g = inp.cuda(), grid.cuda()
    out = Guarded(((N + 1) * (C + 1) * (Ho + 1) * (Wo + 1),), torch.float32)
    ind, gdd = (N, C, Hi, Wi), (N, 2, Ho, Wo)
    for odd in [(N - 1, C, Ho, Wo), (N, C - 1, Ho, Wo), (N, C, Ho - 1, Wo), (N, C, Ho, Wo + 1), (N, C, Wo, Ho),
                (N, C, Ho * Wo)]:  # fmt: skip
        l0 = lib.b200_launch_count()
        st = lib.b200_grid_sampler_enqueue(descs(desc(ind, F32), desc(gdd, F32)), descs(desc(odd, F32)), ptrs(x, g),
                                           ptrs(out.t), None, _lib.current_stream_ptr(), 0, 0, 0)  # fmt: skip
        torch.cuda.synchronize()
        assert out.intact(), odd
        assert st == BAD_PARAM, (odd, st)
        assert lib.b200_launch_count() == l0
    odd = (N, C, Ho, Wo)  # the consistent call still runs and gives the Python op's bits
    st = lib.b200_grid_sampler_enqueue(descs(desc(ind, F32), desc(gdd, F32)), descs(desc(odd, F32)), ptrs(x, g),
                                       ptrs(out.t), None, _lib.current_stream_ptr(), 0, 0, 0)  # fmt: skip
    torch.cuda.synchronize()
    assert st == OK and out.intact()
    assert torch.equal(out.t[: N * C * Ho * Wo].view(odd), bt.grid_sampler(x, g, "bilinear", "zeros", False))


# ---------------------------------------------------------------------------------------------------------------------
# DCN
# name: (N, Ci, H, W, Co, kh, kw, (stride_h, stride_w), (pad_h, pad_w), (dil_h, dil_w), groups, deform_groups), in the
# Python op's (h, w) order. H != W everywhere, and Ho * Wo is never a whole number of the fused kernel's 256- or
# 128-pixel tiles (two cases span more than one).
ASYM_CASES = {
    # fused tcgen05 shapes (C % 64 == 0, Co in {128, 256, 512}, groups = dg = 1, kh * kw <= 9)
    "fused_k1x3_s21_p02_d12": (2, 64, 29, 22, 128, 1, 3, (2, 1), (0, 2), (1, 2), 1, 1),
    "fused_k3x1_s12_p20_d21": (1, 64, 17, 12, 256, 3, 1, (1, 2), (2, 0), (2, 1), 1, 1),
    "fused_k2x3_s21_p02_d12": (2, 128, 11, 19, 128, 2, 3, (2, 1), (0, 2), (1, 2), 1, 1),
    "fused_k3x2_s21": (1, 64, 15, 10, 512, 3, 2, (2, 1), (1, 1), (1, 1), 1, 1),
    "fused_k2x3_p02": (1, 64, 9, 14, 128, 2, 3, (1, 1), (0, 2), (1, 1), 1, 1),
    "fused_k3x1_d12": (1, 64, 20, 16, 128, 3, 1, (1, 1), (1, 0), (1, 2), 1, 1),
    # the same kernels where groups or deformable groups > 1 send them to the generic kernel
    "generic_k1x3_g2_s21_p02_d12": (2, 16, 9, 14, 12, 1, 3, (2, 1), (0, 2), (1, 2), 2, 1),
    "generic_k3x1_dg2_s12_p20_d21": (1, 16, 13, 8, 8, 3, 1, (1, 2), (2, 0), (2, 1), 1, 2),
    "generic_k2x3_g2_dg2_s21_p02_d12": (2, 32, 10, 15, 16, 2, 3, (2, 1), (0, 2), (1, 2), 2, 2),
    "generic_k2x3_dg2_c64_s21_p02_d12": (1, 64, 11, 16, 128, 2, 3, (2, 1), (0, 2), (1, 2), 1, 2),
    # fused-sized channels but kh * kw > 9 (kMaxTaps): the fused path declines, the generic kernel runs
    "generic_k3x5_c64_s21_p02_d12": (1, 64, 12, 19, 128, 3, 5, (2, 1), (0, 2), (1, 2), 1, 1),
    "generic_k5x5_c64_s12_p20_d21": (1, 64, 14, 11, 128, 5, 5, (1, 2), (2, 0), (2, 1), 1, 1),
}
ALL_DCN = list(DCN_CASES) + list(ASYM_CASES)




@functools.lru_cache(maxsize=None)
def dcn_inputs(case):
    """float32 CPU (x, offset, mask, weight, bias) and the geometry as (h, w) pairs, in the Python op's order."""
    if case in DCN_CASES:
        x, off, mask, w, b, kw = make_dcn_inputs(case)
        geo = dict(stride=(kw["stride"],) * 2, padding=(kw["padding"],) * 2, dilation=(kw["dilation"],) * 2,
                   groups=kw["groups"], deform_groups=kw["deform_groups"])  # fmt: skip
        return (x, off, mask, w, b), geo
    N, Ci, H, W, Co, kh, kw, s, p, d, g, dg = ASYM_CASES[case]
    Ho, Wo = odcn.out_size(H, W, kh, kw, s, p, d)
    gen = torch.Generator().manual_seed(7)
    x = torch.randn(N, Ci, H, W, generator=gen)
    off = torch.randn(N, dg * 2 * kh * kw, Ho, Wo, generator=gen) * 1.5
    mask = torch.sigmoid(torch.randn(N, dg * kh * kw, Ho, Wo, generator=gen))
    w = torch.randn(Co, Ci // g, kh, kw, generator=gen) / (Ci // g * kh * kw) ** 0.5
    b = torch.randn(Co, generator=gen)
    return (x, off, mask, w, b), dict(stride=s, padding=p, dilation=d, groups=g, deform_groups=dg)


def quantised(ts):
    """[(q, scale)] of x, offset, mask, weight."""
    return [quantize_per_tensor(t) for t in ts[:4]]


@functools.lru_cache(maxsize=None)
def dcn_oracle(case, kind):
    """The oracle without bias on the case's f32 inputs, their fp16 roundings, or the dequantised int8 tensors. The
    caller adds the bias in float32, as the oracle itself does."""
    ts, geo = dcn_inputs(case)
    if kind == "f32":
        ops = ts[:4]
    elif kind == "f16":
        ops = [t.half().float() for t in ts[:4]]
    else:
        ops = [q.float() * s for q, s in quantised(ts)]
    return odcn.modulated_deformable_conv2d(*(t.numpy() for t in ops), None, **geo)


def with_bias(want, bias):
    return want if bias is None else want + bias.float().numpy()[None, :, None, None]


def form_kind(form):
    return "f32" if form == "f32" else "f16" if form.startswith("f16") else "i8"


def python_op(form, ts, geo, bias, sout=None):
    """The Python op at `geo` for one enqueue form, on the GPU, with the tensors packed as that form requires."""
    x, off, mask, w = ts[:4]
    args = (geo["stride"], geo["padding"], geo["dilation"], geo["groups"], geo["deform_groups"])
    cb = None if bias is None else bias.cuda()
    if form == "f32":
        return bt.modulated_deformable_conv2d(x.cuda(), off.cuda(), mask.cuda(), w.cuda(), cb, *args)
    if form in ("f16", "f16_nobias"):
        return bt.modulated_deformable_conv2d(*(t.half().cuda() for t in (x, off, mask, w)), cb, *args)
    if form == "f16_chw2":
        xh, oh, mh, wh = (t.half() for t in (x, off, mask, w))
        return modulated_deformable_conv2d_chw2(pack_chw(xh, 2).cuda(), pack_chw(oh, 2).cuda(), mh.cuda(),
                                                pack_chw(wh, 2).cuda(), cb, x.shape[1], *args)  # fmt: skip
    (xq, si), (oq, so_), (mq, sm), (wq, sw) = quantised(ts)
    return modulated_deformable_conv2d_int8(pack_chw(xq, 4).cuda(), si, oq.cuda(), so_, mq.cuda(), sm,
                                            pack_chw(wq, 4).cuda(), sw, cb, sout, x.shape[1], *args)  # fmt: skip


def enqueue_operands(form, ts, bias, sout=None, out_hw=None):
    """(input descriptors, output descriptor, device inputs, output shape, output dtype) of one enqueue form. The
    offset / mask / output descriptors claim `out_hw` (default: the offset's own extent)."""
    x, off, mask, w = ts[:4]
    N, C = x.shape[:2]
    Ho, Wo = out_hw or off.shape[2:]
    taps = mask.shape[1]
    xd, od, md, wd = tuple(x.shape), (N, 2 * taps, Ho, Wo), (N, taps, Ho, Wo), tuple(w.shape)
    outd = (N, w.shape[0], Ho, Wo)
    if form in ("f32", "f16", "f16_nobias"):
        tt, dt = (F32, torch.float32) if form == "f32" else (F16, torch.float16)
        dev = [t.to(dt).cuda() for t in (x, off, mask, w)]
        ins, out_desc = [desc(xd, tt), desc(od, tt), desc(md, tt), desc(wd, tt)], desc(outd, tt)
    elif form == "f16_chw2":
        dt = torch.float16
        xh, oh, mh, wh = (t.half() for t in (x, off, mask, w))
        dev = [pack_chw(xh, 2).cuda(), pack_chw(oh, 2).cuda(), mh.cuda(), pack_chw(wh, 2).cuda()]
        ins = [desc(xd, F16, CHW2), desc(od, F16, CHW2), desc(md, F16), desc(wd, F16, CHW2)]
        out_desc = desc(outd, F16)
    else:
        dt = torch.int8
        (xq, si), (oq, so_), (mq, sm), (wq, sw) = quantised(ts)
        dev = [pack_chw(xq, 4).cuda(), oq.cuda(), mq.cuda(), pack_chw(wq, 4).cuda()]
        ins = [desc(xd, I8, CHW4, si), desc(od, I8, LINEAR, so_), desc(md, I8, LINEAR, sm), desc(wd, I8, CHW4, sw)]
        out_desc = desc(outd, I8, LINEAR, sout)
    if bias is not None:
        dev.append(bias.cuda())
        ins.append(desc(tuple(bias.shape), F32 if bias.dtype == torch.float32 else F16))
    return ins, out_desc, dev, outd, dt


def run_dcn_enqueue(ins, out_desc, dev, out, attrs, groups, dg):
    """Allocates exactly b200_dcn_enqueue_workspace_size bytes (256-byte aligned) at the front of a guarded buffer and
    runs the enqueue. Returns (status, workspace guard intact)."""
    lib = _lib.load()
    stride, pad, dil = (ints(*a) for a in attrs)
    in_d = descs(*ins)
    nbytes = lib.b200_dcn_enqueue_workspace_size(in_d, stride, pad, dil, groups, dg)
    assert nbytes > 0
    ws = Guarded((nbytes,), torch.uint8)
    assert ws.t.data_ptr() % 256 == 0
    st = lib.b200_dcn_enqueue(in_d, descs(out_desc), ptrs(*dev), ptrs(out), ws.t.data_ptr(), _lib.current_stream_ptr(),
                              len(ins), stride, pad, dil, groups, dg)  # fmt: skip
    torch.cuda.synchronize()
    return st, ws.intact()


def enqueue_attrs(geo):
    """Plugin attributes {stride, padding, dilation} for a Python-op geometry: element [0] is w, [1] is h."""
    return tuple((geo[k][1], geo[k][0]) for k in ("stride", "padding", "dilation"))


DCN_FORMS = ["f32", "f16", "f16_nobias", "f16_chw2", "i8_f32bias", "i8_f16bias", "i8_nobias"]


def form_bias(form, b):
    if form in ("f16_nobias", "i8_nobias"):
        return None
    return b if form in ("f32", "i8_f32bias") else b.half()


@pytest.mark.parametrize("form", DCN_FORMS)
@pytest.mark.parametrize("case", ALL_DCN)
def test_dcn_enqueue_matches_oracle_and_python_op(case, form):
    """b200_dcn_enqueue in every dtype / format / bias form, against the oracle and, bit for bit, against the Python op
    at the same geometry. The attributes follow the reference plugin's call (modulatedDeformableConv2dPlugin.cpp:
    151-187): element [0] of stride, padding and dilation goes to the launcher's *_w slot and [1] to *_h, and the kernel
    is weight.d[2] (h) x weight.d[3] (w). So enqueue attributes {a0, a1} equal the Python op's stride=(a1, a0), i.e.
    h = a1 and w = a0. This is the intended, reference-compatible behaviour; the ASYM_CASES (H != W, non-square kernels,
    asymmetric attributes) make any other reading fail."""
    ts, geo = dcn_inputs(case)
    bias = form_bias(form, ts[4])
    kind = form_kind(form)
    want = with_bias(dcn_oracle(case, kind), bias)
    sout = float(np.abs(want).max()) / 127.0
    ins, out_desc, dev, outd, dt = enqueue_operands(form, ts, bias, sout)
    out = Guarded(outd, dt)
    st, ws_ok = run_dcn_enqueue(ins, out_desc, dev, out.t, enqueue_attrs(geo), geo["groups"], geo["deform_groups"])
    assert st == OK
    assert ws_ok, "the enqueue wrote past the workspace it asked for"
    assert out.intact(), "the enqueue wrote past its output"
    assert torch.equal(out.t, python_op(form, ts, geo, bias, sout)), "enqueue and Python op disagree"
    if kind == "i8":
        err, tol = np.abs(out.t.cpu().numpy().astype(np.float32) * sout - want).max(), 0.75 * sout
    else:
        err = np.abs(out.t.float().cpu().numpy() - want).max()
        tol = 1e-4 * max(1.0, np.abs(want).max()) if kind == "f32" else fp16_tol(want)
    assert err <= tol, (case, form, err, tol)


def test_dcn_enqueue_attribute_order_is_w_then_h():
    """The same asymmetric layer with its attributes handed over in (h, w) order is a different convolution: with the
    descriptors of the (h, w) geometry the enqueue refuses it, so a shell that serialises the attributes the other way
    round fails loudly instead of computing something else. Read that way, the layer has 13 x 9 output pixels instead
    of 5 x 19; offset, mask and output are sized for both."""
    case = "fused_k2x3_s21_p02_d12"
    (x, off, mask, w, b), geo = dcn_inputs(case)
    N, Co, Ho, Wo = 2, 128, 5, 19
    assert off.shape[2:] == (Ho, Wo)
    hw_order = tuple(geo[k] for k in ("stride", "padding", "dilation"))
    assert hw_order != enqueue_attrs(geo)
    big = [torch.zeros(N, t.shape[1], 13, 19) for t in (off, mask)]
    ins, out_desc, dev, _, dt = enqueue_operands("f16", (x, *big, w), b.half(), out_hw=(Ho, Wo))
    out = Guarded((N, Co, 13, 19), dt)
    l0 = _lib.launch_count()
    st, ws_ok = run_dcn_enqueue(ins, out_desc, dev, out.t, hw_order, 1, 1)
    assert ws_ok and out.intact()
    assert st == BAD_PARAM and _lib.launch_count() == l0


@pytest.mark.parametrize("form", ["f32", "f16", "f16_chw2", "i8_f32bias"])
def test_dcn_enqueue_rejects_descriptors_that_disagree_with_the_attributes(form):
    """The plugin sizes its output from the graph; the launcher re-derives (Ho, Wo) from the attributes, [0] as w. With
    an asymmetric stride on an H != W input the two readings differ: here stride {1, 2} on 13 x 20 is 7 x 20 = 140
    output pixels for the launcher and 13 x 10 = 130 for a graph that reads [0] as h. A kernel run on the launcher's
    reading would read offset / mask and write output past the graph's buffers, so the enqueue must return status 2 and
    launch nothing; likewise for an output, offset, mask or weight descriptor that disagrees in any other dimension.
    Every device buffer is sized for the largest geometry in play, so not even an enqueue without the check can touch
    memory the test does not own."""
    N, C, H, W, Co, k = 1, 8, 13, 20, 128, 3
    attrs = ((1, 2), (1, 1), (1, 1))  # [0] -> w, [1] -> h
    geo = dict(stride=(2, 1), padding=(1, 1), dilation=(1, 1), groups=1, deform_groups=1)  # the Python op's reading
    launcher_hw, graph_hw, big_hw = (7, 20), (13, 10), (13, 20)
    gen = torch.Generator().manual_seed(9)
    x = torch.randn(N, C, H, W, generator=gen)
    off = torch.randn(N, 2 * k * k, *big_hw, generator=gen) * 1.5
    mask = torch.sigmoid(torch.randn(N, k * k, *big_hw, generator=gen))
    w = torch.randn(Co, C, k, k, generator=gen) / (C * k * k) ** 0.5
    b = torch.randn(Co, generator=gen)
    bias = form_bias(form, b)
    sout = 0.05
    lib = _lib.load()
    ts = (x, off, mask, w)
    bad = [(graph_hw, None), (launcher_hw, ("out", 2, 3)), (launcher_hw, ("out", 1, None)),
           (launcher_hw, ("out", 0, None)), (launcher_hw, ("offset", 1, None)), (launcher_hw, ("mask", 3, None)),
           (launcher_hw, ("weight", 1, None))]  # fmt: skip
    for hw, change in bad:
        ins, out_desc, dev, _, dt = enqueue_operands(form, ts, bias, sout, out_hw=hw)
        if change is not None:
            which, i, j = change
            d = {"out": out_desc, "offset": ins[1], "mask": ins[2], "weight": ins[3]}[which].dims.d
            if j is not None:
                d[i], d[j] = d[j], d[i]  # 7 x 20 claimed as 20 x 7: the same number of elements
            else:
                d[i] -= 4 if which == "weight" else 1
        out = Guarded((N + 1, Co, *big_hw), dt)
        l0 = lib.b200_launch_count()
        st, ws_ok = run_dcn_enqueue(ins, out_desc, dev, out.t, attrs, 1, 1)
        assert ws_ok and out.intact(), (form, hw, change)
        assert st == BAD_PARAM, (form, hw, change, st)
        assert lib.b200_launch_count() == l0, (form, hw, change)
    # the consistent call runs, within its buffers, and equals the Python op with stride=(2, 1)
    ts = (x, off[..., : launcher_hw[0], :].contiguous(), mask[..., : launcher_hw[0], :].contiguous(), w)
    ins, out_desc, dev, outd, dt = enqueue_operands(form, ts, bias, sout)
    out = Guarded(outd, dt)
    st, ws_ok = run_dcn_enqueue(ins, out_desc, dev, out.t, attrs, 1, 1)
    assert st == OK and ws_ok and out.intact()
    assert torch.equal(out.t, python_op(form, ts, geo, bias, sout))


# ---------------------------------------------------------------------------------------------------------------------
# Non-square, asymmetric DCN through the Python ops
def _set_fused(on):
    return _lib.load().b200_dcn_set_fused(int(on))


@pytest.mark.parametrize("case", list(ASYM_CASES))
def test_asymmetric_dcn_python_ops_match_oracle(case):
    """fp32; fp16 with the fused tcgen05 path on and off; kCHW2, which must give the linear fp16 bits; int8 on the fused
    and the unfused path. Cases named fused_* are shapes the fused kernels take, generic_* ones they decline (groups or
    deformable groups > 1, or kh * kw above the fused kernel's 9 taps)."""
    ts, geo = dcn_inputs(case)
    x, off, mask, w, b = ts
    want32 = with_bias(dcn_oracle(case, "f32"), b)
    got = python_op("f32", ts, geo, b).cpu().numpy()
    assert np.abs(got - want32).max() <= 1e-4 * max(1.0, np.abs(want32).max())
    want16 = with_bias(dcn_oracle(case, "f16"), b.half())
    bias16 = b.half()
    want8 = with_bias(dcn_oracle(case, "i8"), b)
    sout = float(np.abs(want8).max()) / 127.0
    prev = _set_fused(True)
    try:
        for fused in (True, False):
            _set_fused(fused)
            lin = python_op("f16", ts, geo, bias16)
            err = np.abs(lin.float().cpu().numpy() - want16).max()
            assert err <= fp16_tol(want16), (fused, err, fp16_tol(want16))
            assert torch.equal(python_op("f16_chw2", ts, geo, bias16), lin), fused
            q = python_op("i8_f32bias", ts, geo, b, sout)
            err8 = np.abs(q.cpu().numpy().astype(np.float32) * sout - want8).max()
            assert err8 <= 0.75 * sout, (fused, err8, sout)
    finally:
        _set_fused(prev)


def test_fused_gate_in_python_agrees_with_the_kernel():
    """The Python op sends fp16 DCN to the fused kernel (packed weights, b200_dcn_f16_ex) exactly when the library's
    own gate takes the shape: b200_dcn_pack_weights_f16 accepts it (kh * kw <= kMaxTaps = 9 at C % 64 == 0, Co in
    {128, 256, 512}, groups = dg = 1). Shapes either side of the tap limit, non-square included."""
    mod = importlib.import_module("bevformer_tensorrt_b200.functions.modulated_deformable_conv2d")
    lib = _lib.load()
    N, C, H, W, Co = 1, 64, 9, 12, 128
    calls = []
    orig = mod._forward_fused_f16

    def spy(*a, **k):
        calls.append(1)
        return orig(*a, **k)

    prev = _set_fused(True)
    mod._forward_fused_f16 = spy
    try:
        for kh, kw in [(1, 3), (3, 1), (2, 3), (3, 2), (3, 3), (1, 9), (9, 1), (2, 5), (5, 2), (1, 10), (3, 4), (3, 5),
                       (5, 5)]:  # fmt: skip
            wt = torch.randn(Co, C, kh, kw, device="cuda").half()
            packed = torch.empty_like(wt)
            st = lib.b200_dcn_pack_weights_f16(wt.data_ptr(), packed.data_ptr(), Co, C, kh, kw, _lib.current_stream_ptr())
            assert st == (OK if kh * kw <= 9 else UNSUPPORTED), (kh, kw, st)
            Ho, Wo = H - kh + 1, W - kw + 1
            x = torch.randn(N, C, H, W, device="cuda").half()
            off = torch.randn(N, 2 * kh * kw, Ho, Wo, device="cuda").half()
            mask = torch.rand(N, kh * kw, Ho, Wo, device="cuda").half()
            calls.clear()
            bt.modulated_deformable_conv2d(x, off, mask, wt, None, 1, 0, 1, 1, 1)
            assert len(calls) == (1 if st == OK else 0), (kh, kw)
    finally:
        mod._forward_fused_f16 = orig
        _set_fused(prev)
    torch.cuda.synchronize()
