"""GPU parity tests for multi-scale deformable attention (run on the B200 box: pytest -m gpu).

Bars (BASELINE.json north_star): sampling-index arithmetic bit-exact; values within 1e-3 max-abs (FP16) and 2e-2
(INT8, after multiplying by scale_out); FP32 is held to 1e-5 (the reference's own FP32 op-test bar is mean-abs 1e-5,
test_multi_scale_deformable_attn.py:139-140 — max-abs is stricter).
Checkers: tests/golden (reference Python, and outputs of the reference's own CUDA kernels on a B200),
oracle/msda_oracle.c (CPU restatement).
"""
import ctypes

import numpy as np
import pytest
import torch

import bevformer_tensorrt_b200 as bt
from bevformer_tensorrt_b200 import _lib
from bevformer_tensorrt_b200.functions.multi_scale_deformable_attn import msda_sampling_indices, msda_trace, set_msda_v2
from bevformer_tensorrt_b200.workloads import CONFIGS, MSDAConfig, make_msda_inputs, quantize_per_tensor
from oracle import msda as omsda
from tests.helpers import check_digest, golden_msda_cases, load_golden_msda, load_ref_kernels, sample_index

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
FP16_TOL = 1e-3  # north_star; the default (exact) mode must meet it everywhere
FP16_MIXED_TOL = 1.6e-3  # opt-in mixed mode (fp16 tap weights): documented looser bound
INT8_TOL = 2e-2  # north_star

SMALL = [
    ("small_sca", "U", 11),
    ("small_sca", "edge", 12),
    ("tiny_sca", "U", 13),
    ("cpu_plumbing", "U", 14),
]
EXTRA = {
    "tsa_like": MSDAConfig("tsa_like", 2, 1000, 8, 32, ((30, 30),), 4, 1),
    "decoder_like": MSDAConfig("decoder_like", 1, 900, 8, 32, ((50, 50),), 4, 1),
    "g2": MSDAConfig("g2", 2, 129, 8, 32, ((9, 11), (5, 6)), 8, 2),
    "ragged_tail": MSDAConfig("ragged_tail", 1, 37, 5, 32, ((8, 8), (4, 4)), 4, 1),  # items not a multiple of a block
    "one_pixel": MSDAConfig("one_pixel", 1, 64, 8, 32, ((1, 1), (1, 7), (7, 1)), 4, 4),
    "generic_c20": MSDAConfig("generic_c20", 1, 61, 3, 20, ((7, 9), (4, 5)), 3, 1),  # falls to the generic kernel
    "generic_g3": MSDAConfig("generic_g3", 1, 50, 4, 32, ((6, 6),), 12, 3),
    "many_points": MSDAConfig("many_points", 1, 40, 8, 32, ((10, 12), (5, 6), (3, 3), (2, 2)), 16, 4),
}


def _cfg(name):
    return CONFIGS.get(name) or EXTRA[name]


def _cuda(ts):
    return [t.cuda() for t in ts]


def _oracle_f32(inputs):
    return omsda.msda_f32(*(t.float().numpy() for t in inputs))


# ---------------------------------------------------------------------------------------------------------------
# resident-tail FP16 kernel (csrc/msda_res.cu): the library default behind the FP16 plugin op
# ---------------------------------------------------------------------------------------------------------------
RES_EXTRA = {
    # more (batch, head) pairs than SMs: CTAs walk several pairs and re-stage the tail in between
    "many_pairs": MSDAConfig("many_pairs", 20, 70, 8, 32, ((6, 7), (3, 4), (2, 2)), 8, 4),
    # tail boundary inside the pyramid at every capacity tried below; 3 levels x 8 points
    "three_levels": MSDAConfig("three_levels", 2, 501, 8, 32, ((40, 60), (20, 30), (10, 15)), 8, 2),
}


@pytest.mark.parametrize("cap", [8192, 32768, 131072, 204800])
@pytest.mark.parametrize("name,dist,seed", [("small_sca", "edge", 61), ("small_sca", "U", 62), ("tiny_sca", "G", 63),
                                            ("tsa_like", "edge", 64), ("g2", "edge", 65), ("ragged_tail", "edge", 66),
                                            ("one_pixel", "edge", 67), ("many_pairs", "edge", 68),
                                            ("three_levels", "edge", 69), ("three_levels", "U", 70)])  # fmt: skip
def test_resident_kernel_matches_oracle_and_round1_kernel(name, dist, seed, cap):
    """Same inputs through the resident-tail kernel (coarse levels served from shared memory after TMA staging) at several
    shared-memory capacities — 8 KB: nothing or only the coarsest level resident; 200 KB: everything for the small
    pyramids — and through the round-1 gather kernel. Values within the FP16 bar of the FP32 oracle, and the two kernels
    agree to FP16 rounding (same taps, same FP32 weights; only the order of the two column sums differs); the index
    records traced out of the resident kernel itself are bit-identical to the oracle's."""
    cfg = RES_EXTRA.get(name) or _cfg(name)
    inputs = make_msda_inputs(cfg, dist, seed, torch.float16)
    want = _oracle_f32(inputs)
    dev = _cuda(inputs)
    prev = bt.set_msda_f16_path(True, cap)
    try:
        got = bt.multi_scale_deformable_attn(*dev)
        out_t, rec = msda_trace(*dev)
    finally:
        bt.set_msda_f16_path(prev[0], prev[1])
    prev = bt.set_msda_f16_path(False)
    try:
        r1 = bt.multi_scale_deformable_attn(*dev)
    finally:
        bt.set_msda_f16_path(prev[0])
    err = np.abs(got.float().cpu().numpy() - want).max()
    assert err < FP16_TOL, (name, dist, cap, err)
    assert torch.equal(out_t, got)
    d = (got.float() - r1.float()).abs().max().item()
    assert d <= 2e-3 * max(1.0, float(np.abs(want).max())), (name, cap, d)
    wrec = _want_records(inputs[1], inputs[2].float().numpy(), inputs[3].float().numpy(), cfg)
    assert (rec.cpu().numpy() == wrec).all()


# ---------------------------------------------------------------------------------------------------------------
# golden vectors produced by the reference's own Python code
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", golden_msda_cases())
def test_fp32_matches_reference_golden(path):
    cfg, inputs, want = load_golden_msda(path)
    got = bt.multi_scale_deformable_attn(*_cuda(inputs)).cpu().numpy()
    assert got.shape == want.shape
    assert np.abs(got - want).max() < 2e-5  # golden goes through grid_sample's normalise/un-normalise round trip


# ---------------------------------------------------------------------------------------------------------------
# CPU oracle, seeded inputs
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,dist,seed", SMALL + [(n, "U", 20 + i) for i, n in enumerate(EXTRA)]
                         + [(n, "edge", 40 + i) for i, n in enumerate(EXTRA)])  # fmt: skip
def test_fp32_matches_oracle(name, dist, seed):
    inputs = make_msda_inputs(_cfg(name), dist, seed, torch.float32)
    want = _oracle_f32(inputs)
    for fn in (bt.multi_scale_deformable_attn, bt.multi_scale_deformable_attn2):
        got = fn(*_cuda(inputs)).cpu().numpy()
        assert np.abs(got - want).max() < FP32_TOL, (name, dist, np.abs(got - want).max())


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("name,dist,seed", SMALL + [("tsa_like", "U", 31), ("g2", "edge", 32),
                                                    ("generic_c20", "U", 33), ("many_points", "U", 34)])  # fmt: skip
def test_fp16_matches_oracle(name, dist, seed, mode):
    inputs = make_msda_inputs(_cfg(name), dist, seed, torch.float16)
    want = _oracle_f32(inputs)  # fp32 formulas on the fp16-rounded inputs (SURVEY §7.2-3)
    prev = _lib.load().b200_msda_set_f16_mode(mode)
    try:
        for fn in (bt.multi_scale_deformable_attn, bt.multi_scale_deformable_attn2):
            out = fn(*_cuda(inputs))
            assert out.dtype == torch.float16
            err = np.abs(out.float().cpu().numpy() - want).max()
            assert err < (FP16_TOL if mode == 0 else FP16_MIXED_TOL), (name, dist, mode, err)
    finally:
        _lib.load().b200_msda_set_f16_mode(prev)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("name,dist,seed", [("small_sca", "edge", 51), ("small_sca", "U", 52), ("one_pixel", "edge", 53),
                                            ("tsa_like", "edge", 54), ("tiny_sca", "G", 55)])  # fmt: skip
def test_sampling_indices_bit_exact(name, dist, seed, dtype):
    cfg = _cfg(name)
    value, shapes, ref, off, logits = make_msda_inputs(cfg, dist, seed, dtype)
    _, idx = omsda.msda_f32(value.float().numpy(), shapes.numpy(), ref.float().numpy(), off.float().numpy(),
                            logits.float().numpy(), return_index=True)  # fmt: skip
    rec = msda_sampling_indices(shapes, ref.cuda(), off.cuda(), cfg.num_heads).cpu().numpy()
    want = np.stack([idx["in_range"], idx["h_low"], idx["w_low"], idx["tap_mask"]], -1)
    assert rec.shape == want.shape
    assert (rec == want).all(), f"{(rec != want).any(-1).sum()} of {want[..., 0].size} records differ"
    assert want[..., 0].any() and not want[..., 0].all() or dist == "U"


def _want_records(shapes, ref, off, cfg):
    """Index records of the oracle (oracle/msda_oracle.c restates …Kernel.cu:657-674, :138-172) as int32 [..., 4]."""
    B, Q, M, C = cfg.batch, cfg.num_query, cfg.num_heads, cfg.channels
    NP = cfg.num_levels * cfg.num_points
    dummy_v = np.zeros((B, cfg.spatial_size, M, C), np.float32)
    dummy_w = np.zeros((B, Q, M, NP), np.float32)
    _, idx = omsda.msda_f32(dummy_v, shapes.numpy(), ref, off, dummy_w, return_index=True)
    return np.stack([idx["in_range"], idx["h_low"], idx["w_low"], idx["tap_mask"]], -1)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("name,dist,seed", [("small_sca", "edge", 51), ("small_sca", "U", 52), ("one_pixel", "edge", 53),
                                            ("tsa_like", "edge", 54), ("tiny_sca", "G", 55), ("many_points", "edge", 56),
                                            ("generic_c20", "edge", 57), ("ragged_tail", "edge", 58)])  # fmt: skip
def test_gather_kernel_emits_bit_exact_indices(name, dist, seed, dtype):
    """The records come out of msda_gather_kernel ITSELF (trace instantiation of the production template: same phase A /
    phase C arithmetic, one extra store) — not from a side kernel. `out` of the traced launch must equal the plain
    launch bit for bit, which ties the records to the code path that produced the values."""
    cfg = _cfg(name)
    value, shapes, ref, off, logits = make_msda_inputs(cfg, dist, seed, dtype)
    want = _want_records(shapes, ref.float().numpy(), off.float().numpy(), cfg)
    dev = _cuda([value, shapes, ref, off, logits])
    out_t, rec = msda_trace(*dev)
    out_p = bt.multi_scale_deformable_attn(*dev)
    assert torch.equal(out_t, out_p)
    rec = rec.cpu().numpy()
    assert rec.shape == want.shape
    assert (rec == want).all(), f"{(rec != want).any(-1).sum()} of {want[..., 0].size} records differ"
    assert want[..., 0].any()
    # the stand-alone index kernel agrees as well
    side = msda_sampling_indices(shapes, dev[2], dev[3], cfg.num_heads).cpu().numpy()
    assert (side == want).all()


@pytest.mark.parametrize("dist", ["U", "G"])
def test_gather_kernel_indices_bit_exact_at_base_shapes(dist):
    """BASELINE configs[2] at full size: 61.4 M records from the FP16 production kernel vs the oracle."""
    cfg = CONFIGS["base_sca"]
    value, shapes, ref, off, logits = make_msda_inputs(cfg, dist, 2, torch.float16)
    dev = _cuda([value, shapes, ref, off, logits])
    out_t, rec = msda_trace(*dev)
    assert torch.equal(out_t, bt.multi_scale_deformable_attn(*dev))
    want = _want_records(shapes, ref.float().numpy(), off.float().numpy(), cfg)
    rec = rec.cpu().numpy()
    bad = (rec != want).any(-1).sum()
    assert bad == 0, f"{bad} of {want[..., 0].size} records differ"
    frac = want[..., 0].mean()
    assert (frac > 0.9) if dist == "U" else (0.05 < frac < 0.5)


# ---------------------------------------------------------------------------------------------------------------
# batched launch of the FP32 / FP16 plugin op (visibility scan over 2 / 4 units per warp, csrc/msda.cu UPW)
# ---------------------------------------------------------------------------------------------------------------
BATCH_SHAPES = [(2, False), (4, False), (2, True), (4, True)]


@pytest.fixture
def restore_batch_units():
    prev = bt.get_msda_batch_units()
    yield
    bt.set_msda_batch_units(*prev)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("name,dist,seed", [("small_sca", "edge", 81), ("small_sca", "U", 82), ("tiny_sca", "G", 83),
                                            ("tsa_like", "edge", 84), ("g2", "edge", 85), ("ragged_tail", "edge", 86),
                                            ("one_pixel", "edge", 87), ("many_points", "edge", 88),
                                            ("cpu_plumbing", "U", 89), ("decoder_like", "edge", 90)])  # fmt: skip
def test_batched_launch_is_bit_identical(name, dist, seed, dtype, restore_batch_units):
    """Every launch shape of the plugin op (1 / 2 / 4 units per warp, neighbouring or grid-strided) must give the same
    bytes: same item groups per warp, same arithmetic, only the order in which a warp meets its groups changes. The
    traced launch follows the same switch, so the index records of the batched kernel are checked against the oracle
    too. Shapes outside the batched envelope (heads that do not divide a block, > 2 rounds) silently take the
    one-unit grid and must of course agree as well."""
    cfg = _cfg(name)
    inputs = make_msda_inputs(cfg, dist, seed, dtype)
    dev = _cuda(inputs)
    bt.set_msda_batch_units(1)
    base = bt.multi_scale_deformable_attn(*dev)
    err = np.abs(base.float().cpu().numpy() - _oracle_f32(inputs)).max()
    assert err < (FP32_TOL if dtype == torch.float32 else FP16_TOL)
    want = _want_records(inputs[1], inputs[2].float().numpy(), inputs[3].float().numpy(), cfg)
    for units, strided in BATCH_SHAPES:
        bt.set_msda_batch_units(units, strided)
        assert bt.get_msda_batch_units() == (units, strided)
        got = bt.multi_scale_deformable_attn(*dev)
        assert torch.equal(got, base), (name, units, strided, (got.float() - base.float()).abs().max().item())
        out_t, rec = msda_trace(*dev)
        assert torch.equal(out_t, base), (name, units, strided)
        assert (rec.cpu().numpy() == want).all(), (name, units, strided)


@pytest.mark.parametrize("dist", ["U", "G"])
def test_batched_launch_bit_identical_at_base_shapes(dist, restore_batch_units):
    """BASELINE configs[2] at full size, FP16 and FP32, against the one-unit grid (itself checked against the
    reference's own kernel and the oracle elsewhere in this file); the FP16 index records of the 4-unit kernel against
    the oracle."""
    cfg = CONFIGS["base_sca"]
    inputs = make_msda_inputs(cfg, dist, 2, torch.float16)
    dev = _cuda(inputs)
    dev32 = [t.float() if t.is_floating_point() else t for t in dev]
    bt.set_msda_batch_units(1)
    base16, base32 = bt.multi_scale_deformable_attn(*dev), bt.multi_scale_deformable_attn(*dev32)
    for units, strided in BATCH_SHAPES:
        bt.set_msda_batch_units(units, strided)
        assert torch.equal(bt.multi_scale_deformable_attn(*dev), base16), (units, strided)
        assert torch.equal(bt.multi_scale_deformable_attn(*dev32), base32), (units, strided)
    bt.set_msda_batch_units(4, False)
    out_t, rec = msda_trace(*dev)
    assert torch.equal(out_t, base16)
    want = _want_records(inputs[1], inputs[2].float().numpy(), inputs[3].float().numpy(), cfg)
    assert (rec.cpu().numpy() != want).any(-1).sum() == 0


@pytest.mark.parametrize("ref_dtype", [torch.float32, torch.float16])
def test_int8_gather_kernel_indices_bit_exact(ref_dtype):
    cfg = _cfg("small_sca")
    value, shapes, ref, off, logits = make_msda_inputs(cfg, "edge", 59, torch.float32)
    vq, sv = quantize_per_tensor(value)
    oq, so = quantize_per_tensor(off)
    wq, sw = quantize_per_tensor(logits)
    ref = ref.to(ref_dtype)
    # offsets are dequantised as float(q) * scale in fp32, then fused with ref * size (…Kernel.cu:916-921)
    off_real = oq.numpy().astype(np.float32) * np.float32(so)
    want = _want_records(shapes, ref.float().numpy(), off_real, cfg)
    out_t, rec = msda_trace(vq.cuda(), shapes.cuda(), ref.cuda(), oq.cuda(), wq.cuda(), scales=(sv, so, sw, 0.02))
    out_p = bt.multi_scale_deformable_attn_int8(vq.cuda(), sv, shapes.cuda(), ref.cuda(), oq.cuda(), so, wq.cuda(), sw, 0.02)
    assert torch.equal(out_t, out_p)
    assert (rec.cpu().numpy() == want).all()


# ---------------------------------------------------------------------------------------------------------------
# INT8
# ---------------------------------------------------------------------------------------------------------------
def _quantised(cfg, dist, seed, ref_dtype, want_real=True):
    value, shapes, ref, off, logits = make_msda_inputs(cfg, dist, seed, torch.float32)
    vq, sv = quantize_per_tensor(value)
    oq, so = quantize_per_tensor(off)
    wq, sw = quantize_per_tensor(logits)
    ref = ref.to(ref_dtype)
    if not want_real:  # kernel-against-kernel comparisons at sizes the CPU oracle does not finish in seconds
        return (vq, sv, shapes, ref, oq, so, wq, sw, 1.6 / 127.0), None
    real = omsda.msda_f32(vq.float().numpy() * sv, shapes.numpy(), ref.float().numpy(), oq.float().numpy() * so,
                          wq.float().numpy() * sw)  # fmt: skip
    sout = float(np.abs(real).max()) / 127.0
    return (vq, sv, shapes, ref, oq, so, wq, sw, sout), real


@pytest.mark.parametrize("ref_dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("name,dist,seed", [("small_sca", "U", 61), ("small_sca", "edge", 62), ("tiny_sca", "U", 63),
                                            ("tsa_like", "U", 64), ("many_points", "U", 65)])  # fmt: skip
def test_int8_matches_dequant_oracle(name, dist, seed, ref_dtype):
    (vq, sv, shapes, ref, oq, so, wq, sw, sout), real = _quantised(_cfg(name), dist, seed, ref_dtype)
    got = bt.multi_scale_deformable_attn_int8(vq.cuda(), sv, shapes, ref.cuda(), oq.cuda(), so, wq.cuda(), sw, sout)
    assert got.dtype == torch.int8
    got = got.cpu().numpy()
    # (1) north_star bar: dequantised output vs the fp32 formulas on dequantised inputs
    assert np.abs(got.astype(np.float32) * sout - real).max() < INT8_TOL
    # (2) against the oracle's own requantisation: identical up to 1 LSB on rounding ties
    want_q = omsda.msda_i8_dequant(vq.numpy(), sv, shapes.numpy(), ref.float().numpy(), oq.numpy(), so, wq.numpy(), sw,
                                   sout)  # fmt: skip
    diff = np.abs(got.astype(np.int32) - want_q.astype(np.int32))
    # (fp16 tap weights in the INT8 kernel move a few results across a rounding boundary)
    assert diff.max() <= 1 and (diff != 0).mean() < 0.02, (diff.max(), (diff != 0).mean())


# ---------------------------------------------------------------------------------------------------------------
# the reference's own CUDA kernels, run on a B200 (tests/golden/ref_kernels_msda.npz, make_golden_ref_kernels.py):
# outputs too large for a fixture as a fixed, seeded sample; the reference's own errors over every element as numbers
# ---------------------------------------------------------------------------------------------------------------
REFK = load_ref_kernels("msda")


def _at_sample(t, k=2048):
    """Elements of t at the positions of the fixture's seeded sample of about k elements, on the CPU."""
    flat = t.reshape(-1)
    return flat[torch.from_numpy(sample_index(flat.numel(), k)).to(flat.device)].cpu()


@pytest.mark.parametrize("name,dist,seed", [("small_sca", "edge", 71), ("tiny_sca", "U", 72), ("tsa_like", "U", 73)])
def test_fp32_matches_reference_kernel(name, dist, seed):
    host = make_msda_inputs(_cfg(name), dist, seed, torch.float32)
    key = f"fp32_{name}_{dist}_{seed}"
    check_digest(REFK, key, *host)
    got = bt.multi_scale_deformable_attn(*_cuda(host))
    assert (_at_sample(got) - torch.from_numpy(REFK[key])).abs().max().item() < FP32_TOL


def test_base_shapes_fp32_against_reference_kernel_full_size():
    """BASELINE configs[2] at full size, GPU vs GPU."""
    host = make_msda_inputs(CONFIGS["base_sca"], "U", 0, torch.float32)
    check_digest(REFK, "fp32_base_U_0", *host)
    got = bt.multi_scale_deformable_attn(*_cuda(host))
    assert got.shape == (6, 40000, 8, 32)
    want = REFK["fp32_base_U_0"]
    assert (_at_sample(got, 4096) - torch.from_numpy(want)).abs().max().item() < FP32_TOL


@pytest.mark.parametrize("dist", ["U", "G"])
def test_base_shapes_fp16_within_tolerance_of_fp32_reference_kernel(dist):
    """FP16 I/O at full size vs the reference FP32 kernel run on the same (fp16-rounded) inputs; also reports how far
    the reference's own __half / __half2 kernels are from that truth (they do the coordinate math in half)."""
    h = make_msda_inputs(CONFIGS["base_sca"], dist, 1, torch.float16)
    key = f"fp16_base_{dist}_1"
    check_digest(REFK, key, *h)
    hin = _cuda(h)
    truth = torch.from_numpy(REFK[f"{key}_truth"])
    for mode in (0, 1):
        prev = _lib.load().b200_msda_set_f16_mode(mode)
        try:
            got = bt.multi_scale_deformable_attn(*hin).float()
        finally:
            _lib.load().b200_msda_set_f16_mode(prev)
        err = (_at_sample(got) - truth).abs().max().item()
        print(f"\n[base {dist}] ours fp16 mode {mode}: max-abs vs fp32 reference kernel = {err:.3e}")
        assert err < (FP16_TOL if mode == 0 else FP16_MIXED_TOL)
    for variant in ("f16", "f16_h2"):
        e = float(REFK[f"{key}_err_{variant}"])
        print(f"[base {dist}] reference {variant} kernel: max-abs vs its own fp32 kernel = {e:.3e}")


@pytest.mark.parametrize("ref_dtype", [torch.float32, torch.float16])
def test_int8_vs_reference_int8_kernel(ref_dtype):
    """Informational + sanity: the reference INT8 kernels quantise intermediates (SURVEY A.4), so they differ from the
    in-register-dequant definition by O(1 LSB); both must sit within the INT8 bar of the fp32 truth."""
    (vq, sv, shapes, ref, oq, so, wq, sw, sout), real = _quantised(_cfg("small_sca"), "U", 81, ref_dtype)
    key = f"i8_small_sca_U_81_{str(ref_dtype).split('.')[-1]}"
    check_digest(REFK, key, vq, shapes, ref, oq, wq)
    assert sout == float(REFK[f"{key}_sout"])
    args = (vq.cuda(), sv, shapes.cuda(), ref.cuda(), oq.cuda(), so, wq.cuda(), sw, sout)
    ours = bt.multi_scale_deformable_attn_int8(*args).cpu().numpy().astype(np.float32) * sout
    e_ours, e_theirs = np.abs(ours - real).max(), float(REFK[f"{key}_err"])
    print(f"\n[int8 {ref_dtype}] ours {e_ours:.4f}  reference kernel {e_theirs:.4f}  (scale_out {sout:.4f})")
    assert e_ours < INT8_TOL
    assert e_ours <= e_theirs + 1e-6  # dequantising in registers can only be closer to the fp32 truth
    if ref_dtype == torch.float32:  # the CPU emulation of the quantised-intermediate kernel pins oracle <-> reference
        emu = omsda.msda_i8_refemu(vq.numpy(), sv, shapes.numpy(), ref.float().numpy(), oq.numpy(), so, wq.numpy(), sw,
                                   sout)  # fmt: skip
        theirs = REFK[key].astype(np.float32)
        d = np.abs(emu.reshape(-1)[sample_index(emu.size, 4096)].astype(np.float32) - theirs)
        assert d.max() <= 1.0 and (d != 0).mean() < 0.02, (d.max(), (d != 0).mean())


@pytest.mark.parametrize("ref_dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("dist", ["U", "G"])
def test_base_shapes_int8_config4(dist, ref_dtype):
    """BASELINE configs[3] (INT8 per-tensor PTQ at base shapes, [6,40000,8,32]):
    (1) ours vs the fp32 truth = the reference's own FP32 kernel (…Kernel.cu:611-688) on the dequantised inputs: the
        north_star INT8 bar 2e-2 max-abs after x scale_out, on the fixture's sample of that truth and, over every element,
        against this library's FP32 kernel on the same inputs (itself held to 1e-5 of the reference's on the sample);
    (2) the reference's own INT8 kernels ms_deformable_im2col_cuda_int8<float|__half2> (…Kernel.cu:1172-1218) on the
        same quantised tensors: theirs quantise intermediates, so ours must be at least as close to the truth;
    (3) ours vs the CPU dequant oracle's requantisation: at most 1 LSB apart, on < 2 % of the elements."""
    cfg = CONFIGS["base_sca"]
    value, shapes, ref, off, logits = make_msda_inputs(cfg, dist, 3, torch.float32)
    vq, sv = quantize_per_tensor(value)
    oq, so = quantize_per_tensor(off)
    wq, sw = quantize_per_tensor(logits)
    ref = ref.to(ref_dtype)
    key = f"i8_base_{dist}_3_{str(ref_dtype).split('.')[-1]}"
    check_digest(REFK, key, vq, shapes, ref, oq, wq)
    dq = [vq.cuda().float() * sv, shapes.cuda(), ref.cuda().float(), oq.cuda().float() * so, wq.cuda().float() * sw]
    truth = torch.from_numpy(REFK[f"{key}_truth"])
    ours32 = bt.multi_scale_deformable_attn(*dq)
    assert (_at_sample(ours32) - truth).abs().max().item() < FP32_TOL
    sout = float(REFK[f"{key}_truth_amax"]) / 127.0
    args = (vq.cuda(), sv, shapes.cuda(), ref.cuda(), oq.cuda(), so, wq.cuda(), sw, sout)
    ours_q = bt.multi_scale_deformable_attn_int8(*args)
    e_ours = (_at_sample(ours_q).float() * sout - truth).abs().max().item()
    e_ours_all = (ours_q.float() * sout - ours32).abs().max().item()
    e_theirs = float(REFK[f"{key}_err"])
    print(f"\n[base int8 {dist} ref {ref_dtype}] ours {e_ours_all:.4e}  reference int8 kernel {e_theirs:.4e}  scale_out {sout:.4e}")
    assert e_ours < INT8_TOL and e_ours_all < INT8_TOL
    assert e_ours <= e_theirs + 1e-6 and e_ours_all <= e_theirs + FP32_TOL
    assert ours_q.float().abs().max().item() >= 100  # the output scale is actually used
    want_q = omsda.msda_i8_dequant(vq.numpy(), sv, shapes.numpy(), ref.float().numpy(), oq.numpy(), so, wq.numpy(), sw, sout)
    diff = np.abs(ours_q.cpu().numpy().astype(np.int32) - want_q.astype(np.int32))
    assert diff.max() <= 1 and (diff != 0).mean() < 0.02, (diff.max(), (diff != 0).mean())


# ---------------------------------------------------------------------------------------------------------------
# size-independent properties at full BASELINE size
# ---------------------------------------------------------------------------------------------------------------
def test_base_shapes_properties_fp32():
    value, shapes, ref, off, logits = _cuda(make_msda_inputs(CONFIGS["base_sca"], "U", 5, torch.float32))
    f = bt.multi_scale_deformable_attn
    out = f(value, shapes, ref, off, logits)
    # softmax shift invariance
    out_shift = f(value, shapes, ref, off, logits + 3.0)
    assert (out - out_shift).abs().max().item() < 5e-6
    # linearity in value
    v2 = torch.randn_like(value)
    lin = f(2.0 * value + v2, shapes, ref, off, logits)
    assert (lin - (2.0 * out + f(v2, shapes, ref, off, logits))).abs().max().item() < 2e-5
    # a constant image sampled strictly inside returns the constant: shrink refs/offsets so no tap leaves the image
    ones = torch.ones_like(value)
    inner_ref = ref * 0.5 + 0.25
    small_off = off.clamp(-1.0, 1.0)
    const = f(ones, shapes, inner_ref, small_off, logits)
    assert (const - 1.0).abs().max().item() < 1e-5
    # everything out of range -> exact zeros
    far = f(value, shapes, ref + 5.0, off, logits)
    assert far.abs().max().item() == 0.0


def test_base_shapes_fp16_vs_fp32_kernel_full_size():
    h = make_msda_inputs(CONFIGS["base_sca"], "U", 6, torch.float16)
    hin = _cuda(h)
    fin = [t.float() if t.is_floating_point() else t for t in hin]
    truth = bt.multi_scale_deformable_attn(*fin)
    for mode in (0, 1):
        prev = _lib.load().b200_msda_set_f16_mode(mode)
        try:
            got = bt.multi_scale_deformable_attn(*hin).float()
        finally:
            _lib.load().b200_msda_set_f16_mode(prev)
        assert (got - truth).abs().max().item() < (FP16_TOL if mode == 0 else FP16_MIXED_TOL)


# ---------------------------------------------------------------------------------------------------------------
# second-generation INT8 path (csrc/msda_v2.cu) against the oracle and the round-1 kernel
# ---------------------------------------------------------------------------------------------------------------
V2_CASES = {
    "v2_odd_levels": MSDAConfig("v2_odd_levels", 2, 257, 8, 32, ((13, 21), (7, 11), (4, 6), (1, 3)), 8, 4),  # odd H and W, 1-row level
    "v2_two_levels": MSDAConfig("v2_two_levels", 1, 100, 8, 32, ((9, 70), (5, 129)), 8, 2),  # W > one 64-column pack tile
    "v2_np16": MSDAConfig("v2_np16", 3, 77, 3, 32, ((6, 6), (3, 3)), 8, 1),  # 16 points: half of the owner lanes idle
    "v2_np24": MSDAConfig("v2_np24", 1, 50, 5, 32, ((8, 9), (4, 5), (2, 3)), 8, 4),
}


@pytest.fixture(params=[4096, 131072])
def i8_resident_bytes(request):
    """Shared memory the INT8 gather kernel may keep resident: 4 KB (at most the coarsest level of the small pyramids:
    most samples take the global path) and the 128 KB default (small pyramids entirely resident)."""
    lib = _lib.load()
    prev = lib.b200_msda_set_i8_resident_bytes(request.param)
    yield request.param
    lib.b200_msda_set_i8_resident_bytes(prev)


@pytest.mark.parametrize("ref_dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("name,dist,seed", [("small_sca", "U", 111), ("small_sca", "edge", 112), ("v2_odd_levels", "edge", 113),
                                            ("v2_two_levels", "edge", 114), ("v2_np16", "U", 115), ("v2_np24", "edge", 116),
                                            ("many_pairs", "edge", 117)])  # fmt: skip
def test_v2_int8_matches_oracle_and_round1_kernel(name, dist, seed, ref_dtype, i8_resident_bytes):
    cfg = CONFIGS.get(name) or V2_CASES.get(name) or RES_EXTRA[name]
    lib = _lib.load()
    assert lib.b200_msda_i8_workspace_size(cfg.batch, cfg.spatial_size, cfg.num_heads, 32, cfg.num_levels, cfg.num_points,
                                           cfg.points_per_group) > 0  # these shapes are inside the v2 envelope
    (vq, sv, shapes, ref, oq, so, wq, sw, sout), real = _quantised(cfg, dist, seed, ref_dtype)
    args = (vq.cuda(), sv, shapes.cuda(), ref.cuda(), oq.cuda(), so, wq.cuda(), sw, sout)
    n0 = _lib.launch_count()
    got_t = bt.multi_scale_deformable_attn_int8(*args)
    assert _lib.launch_count() == n0 + 2  # pack + gather
    got = got_t.cpu().numpy()
    assert np.abs(got.astype(np.float32) * sout - real).max() < INT8_TOL
    want_q = omsda.msda_i8_dequant(vq.numpy(), sv, shapes.numpy(), ref.float().numpy(), oq.numpy(), so, wq.numpy(), sw, sout)
    diff = np.abs(got.astype(np.int32) - want_q.astype(np.int32))
    assert diff.max() <= 1 and (diff != 0).mean() < 0.02, (diff.max(), (diff != 0).mean())
    # the v2 gather kernel's own index records, bit-exact
    out_t, rec = msda_trace(args[0], args[2], args[3], args[4], args[6], scales=(sv, so, sw, sout))
    assert torch.equal(out_t, got_t)
    off_real = oq.numpy().astype(np.float32) * np.float32(so)
    assert (rec.cpu().numpy() == _want_records(shapes, ref.float().numpy(), off_real, cfg)).all()
    # round-1 kernel on the same tensors: at most 1 LSB apart on a few elements
    prev = set_msda_v2(False)
    try:
        n0 = _lib.launch_count()
        v1 = bt.multi_scale_deformable_attn_int8(*args).cpu().numpy()
        assert _lib.launch_count() == n0 + 1
    finally:
        set_msda_v2(prev)
    d1 = np.abs(v1.astype(np.int32) - got.astype(np.int32))
    assert d1.max() <= 1 and (d1 != 0).mean() < 0.03


@pytest.mark.parametrize("ref_dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("name,dist,seed", [("small_sca", "edge", 121), ("tiny_sca", "G", 122), ("v2_odd_levels", "edge", 123),
                                            ("v2_np16", "U", 124), ("many_pairs", "edge", 125), ("g2", "edge", 126)])  # fmt: skip
def test_v2_int8_batched_walk_is_bit_identical(name, dist, seed, ref_dtype, i8_resident_bytes, restore_batch_units):
    """The INT8 gather kernel walking 2 / 4 query blocks at a time (visibility scan staged through the warp's record
    area by cp.async) against the one-block walk: same bytes, and the index records traced out of the batched kernel
    itself are the oracle's."""
    cfg = CONFIGS.get(name) or V2_CASES.get(name) or RES_EXTRA.get(name) or EXTRA[name]
    (vq, sv, shapes, ref, oq, so, wq, sw, sout), _ = _quantised(cfg, dist, seed, ref_dtype)
    args = (vq.cuda(), sv, shapes.cuda(), ref.cuda(), oq.cuda(), so, wq.cuda(), sw, sout)
    bt.set_msda_batch_units(1)
    base = bt.multi_scale_deformable_attn_int8(*args)
    off_real = oq.numpy().astype(np.float32) * np.float32(so)
    want = _want_records(shapes, ref.float().numpy(), off_real, cfg)
    for units in (2, 4):
        bt.set_msda_batch_units(units)
        assert torch.equal(bt.multi_scale_deformable_attn_int8(*args), base), (name, units)
        out_t, rec = msda_trace(args[0], args[2], args[3], args[4], args[6], scales=(sv, so, sw, sout))
        assert torch.equal(out_t, base), (name, units)
        assert (rec.cpu().numpy() == want).all(), (name, units)


@pytest.mark.parametrize("dist", ["U", "G"])
def test_v2_int8_batched_walk_bit_identical_at_base_shapes(dist, restore_batch_units):
    """BASELINE configs[3] tensors (INT8 at base shapes), half and float reference points."""
    cfg = CONFIGS["base_sca"]
    for ref_dtype in (torch.float16, torch.float32):
        (vq, sv, shapes, ref, oq, so, wq, sw, sout), _ = _quantised(cfg, dist, 4, ref_dtype, want_real=False)
        args = (vq.cuda(), sv, shapes.cuda(), ref.cuda(), oq.cuda(), so, wq.cuda(), sw, sout)
        bt.set_msda_batch_units(1)
        base = bt.multi_scale_deformable_attn_int8(*args)
        for units in (2, 4):
            bt.set_msda_batch_units(units)
            assert torch.equal(bt.multi_scale_deformable_attn_int8(*args), base), (dist, ref_dtype, units)


def test_v2_envelope_and_fallback():
    lib = _lib.load()
    assert lib.b200_msda_i8_workspace_size(2, 40000, 8, 32, 1, 4, 1) == 0  # TSA: 4 points
    assert lib.b200_msda_i8_workspace_size(1, 100, 8, 20, 4, 8, 4) == 0  # channels != 32
    cfg = EXTRA["many_points"]  # 64 points: outside the envelope, the op silently takes the round-1 kernel
    (vq, sv, shapes, ref, oq, so, wq, sw, sout), real = _quantised(cfg, "U", 7, torch.float16)
    n0 = _lib.launch_count()
    out = bt.multi_scale_deformable_attn_int8(vq.cuda(), sv, shapes, ref.cuda(), oq.cuda(), so, wq.cuda(), sw, sout)
    assert _lib.launch_count() == n0 + 1
    assert np.abs(out.cpu().numpy().astype(np.float32) * sout - real).max() < INT8_TOL
    # a too-small workspace is an error, not a silent overrun
    cfg = _cfg("small_sca")
    (vq, sv, shapes, ref, oq, so, wq, sw, sout), _ = _quantised(cfg, "U", 8, torch.float16)
    t = [x.cuda() for x in (vq, shapes, ref, oq, wq)]
    out = torch.empty(cfg.batch, cfg.num_query, cfg.num_heads, 32, dtype=torch.int8, device="cuda")
    ws = torch.empty(1024, dtype=torch.uint8, device="cuda")
    st = lib.b200_msda_i8_ws(t[0].data_ptr(), sv, t[1].data_ptr(), t[2].data_ptr(), 1, t[3].data_ptr(), so, t[4].data_ptr(), sw,
                             cfg.batch, cfg.spatial_size, cfg.num_heads, 32, cfg.num_levels, cfg.num_query, cfg.num_points,
                             cfg.points_per_group, out.data_ptr(), sout, ws.data_ptr(), ws.numel(), None,
                             _lib.current_stream_ptr())  # fmt: skip
    assert st == 2


# ---------------------------------------------------------------------------------------------------------------
# boundary behaviour
# ---------------------------------------------------------------------------------------------------------------
def test_plugin_enqueue_entry_matches_function():
    cfg = _cfg("small_sca")
    value, shapes, ref, off, logits = _cuda(make_msda_inputs(cfg, "U", 91, torch.float16))
    want = bt.multi_scale_deformable_attn(value, shapes, ref, off, logits)
    lib = _lib.load()

    def desc(t, ttype, scale=1.0):
        d = _lib.TensorDesc()
        d.dims.nbDims = t.dim()
        for i, s in enumerate(t.shape):
            d.dims.d[i] = s
        d.type, d.format, d.scale = ttype, 0, scale
        return d

    out = torch.empty_like(want)
    ins = [value, shapes, ref, off, logits]
    in_desc = (_lib.TensorDesc * 5)(desc(value, 1), desc(shapes, 3), desc(ref, 1), desc(off, 1), desc(logits, 1))
    out_desc = (_lib.TensorDesc * 1)(desc(out, 1))
    in_ptrs = (ctypes.c_void_p * 5)(*[t.data_ptr() for t in ins])
    out_ptrs = (ctypes.c_void_p * 1)(out.data_ptr())
    for pos in range(6):
        io = (_lib.TensorDesc * 6)(*in_desc, out_desc[0])
        assert lib.b200_msda_supports_format(pos, io, 5, 1) == 1
    st = lib.b200_msda_enqueue(in_desc, out_desc, in_ptrs, out_ptrs, None, _lib.current_stream_ptr(), 1)
    assert st == 0
    torch.cuda.synchronize()
    assert torch.equal(out, want)
    assert lib.b200_msda_enqueue_workspace_size(in_desc) == 0  # FP16: round-1 kernel, 0 bytes like the reference
    # INT8: workspace == NULL runs the round-1 kernel (the reference's 0-byte workspace, …Plugin.cpp:64-69), the workspace
    # getWorkspaceSize asks for selects the second-generation kernels (what the Python op runs)
    (vq, sv, shq, rq, oq, so, wq, sw, sout), _ = _quantised(cfg, "U", 191, torch.float16)
    qt = [vq.cuda(), shq.cuda(), rq.cuda(), oq.cuda(), wq.cuda()]
    want8 = bt.multi_scale_deformable_attn_int8(qt[0], sv, qt[1], qt[2], qt[3], so, qt[4], sw, sout)
    out8 = torch.empty_like(want8)
    d8 = (_lib.TensorDesc * 5)(desc(qt[0], 2, sv), desc(qt[1], 3), desc(qt[2], 1), desc(qt[3], 2, so), desc(qt[4], 2, sw))
    o8 = (_lib.TensorDesc * 1)(desc(out8, 2, sout))
    p8 = (ctypes.c_void_p * 5)(*[t.data_ptr() for t in qt])
    q8 = (ctypes.c_void_p * 1)(out8.data_ptr())
    nbytes = lib.b200_msda_enqueue_workspace_size(d8)
    assert nbytes == lib.b200_msda_i8_workspace_size(*vq.shape, shq.shape[0], cfg.num_points, cfg.points_per_group) > 0
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    assert lib.b200_msda_enqueue(d8, o8, p8, q8, ws.data_ptr(), _lib.current_stream_ptr(), 0) == 0
    torch.cuda.synchronize()
    assert torch.equal(out8, want8)
    prev = set_msda_v2(False)
    try:
        want8_r1 = bt.multi_scale_deformable_attn_int8(qt[0], sv, qt[1], qt[2], qt[3], so, qt[4], sw, sout)
    finally:
        set_msda_v2(prev)
    assert lib.b200_msda_enqueue(d8, o8, p8, q8, None, _lib.current_stream_ptr(), 0) == 0
    torch.cuda.synchronize()
    assert torch.equal(out8, want8_r1)
    in_desc[0].type = 3  # int32 value: unsupported dtype -> 1, like the reference's enqueue
    assert lib.b200_msda_enqueue(in_desc, out_desc, in_ptrs, out_ptrs, None, _lib.current_stream_ptr(), 0) == 1


def test_error_behaviour():
    cfg = _cfg("small_sca")
    value, shapes, ref, off, logits = make_msda_inputs(cfg, "U", 92, torch.float32)
    with pytest.raises(AssertionError):
        bt.multi_scale_deformable_attn(value, shapes, ref, off, logits)  # CPU tensor: `assert value.is_cuda`
    cu = _cuda([value, shapes, ref, off, logits])
    with pytest.raises(_lib.B200OpsError):
        bt.multi_scale_deformable_attn(cu[0].double(), *cu[1:])
    with pytest.raises(ValueError):
        bt.multi_scale_deformable_attn(cu[0], cu[1], cu[2], cu[3][..., :-2], cu[4])
    lib = _lib.load()
    assert lib.b200_msda_f32(None, None, None, None, None, 1, 1, 1, 32, 1, 1, 4, 1, None, None) == 2
    n0 = _lib.launch_count()
    bt.multi_scale_deformable_attn(*cu)
    assert _lib.launch_count() == n0 + 1


def test_noncontiguous_and_int64_shapes():
    cfg = _cfg("small_sca")
    value, shapes, ref, off, logits = _cuda(make_msda_inputs(cfg, "U", 93, torch.float32))
    want = bt.multi_scale_deformable_attn(value, shapes, ref, off, logits)
    v_nc = value.permute(0, 2, 1, 3).contiguous().permute(0, 2, 1, 3)
    got = bt.multi_scale_deformable_attn(v_nc, shapes.long(), ref, off, logits)
    assert torch.equal(got, want)


# ---------------------------------------------------------------------------------------------------------------
# fused SCA sampling (MSDA + bev_mask camera-sum), SURVEY §8(f)-1
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,tol", [(torch.float32, 2e-5), (torch.float16, 1e-3)])
@pytest.mark.parametrize("name,dist", [("tiny_sca", "G"), ("small_sca", "edge")])
def test_fused_sca_matches_masked_camera_sum_of_oracle(name, dist, dtype, tol):
    from bevformer_tensorrt_b200.workloads import bev_reference_points_cam, camera_ring_lidar2img

    cfg = _cfg(name)
    inputs = make_msda_inputs(cfg, dist, 101, dtype)
    if cfg.bev_hw[0] * cfg.bev_hw[1] == cfg.num_query:
        _, mask = bev_reference_points_cam(cfg.bev_hw, camera_ring_lidar2img(cfg.batch))
    else:
        mask = (torch.rand(cfg.batch, cfg.num_query, 1, generator=torch.Generator().manual_seed(3)) > 0.4).float()
    per_cam = torch.from_numpy(_oracle_f32(inputs))  # [B,Q,M,C]
    want = (per_cam.reshape(cfg.batch, cfg.num_query, -1) * mask).sum(0)  # spatial_cross_attention.py:270
    got = bt.multi_scale_deformable_attn_sca(*_cuda(inputs), mask.cuda())
    assert got.dtype == torch.float32 and got.shape == want.shape
    assert (got.cpu() - want).abs().max().item() < tol
    # += semantics on a caller-provided accumulator
    acc = torch.ones_like(got)
    bt.multi_scale_deformable_attn_sca(*_cuda(inputs), mask.cuda(), acc)
    assert (acc - 1.0 - got).abs().max().item() < 1e-6


def test_fused_sca_base_shapes_vs_plugin_op():
    from bevformer_tensorrt_b200.workloads import bev_reference_points_cam, camera_ring_lidar2img

    cfg = CONFIGS["base_sca"]
    ins = _cuda(make_msda_inputs(cfg, "G", 7, torch.float16))
    _, mask = bev_reference_points_cam(cfg.bev_hw, camera_ring_lidar2img(6))
    mask = mask.cuda()
    fin = [t.float() if t.is_floating_point() else t for t in ins]
    want = (bt.multi_scale_deformable_attn(*fin).reshape(6, cfg.num_query, -1) * mask).sum(0)
    got = bt.multi_scale_deformable_attn_sca(*ins, mask)
    assert (got - want).abs().max().item() < 1e-3
    assert got.abs().max().item() > 0.1


# ---------------------------------------------------------------------------------------------------------------
# camera-shared fused SCA: offsets / logits passed once (the reference repeats the query per camera,
# spatial_cross_attention.py:254, so the plugin's [bs, ...] offsets / logits are bs identical copies)
# ---------------------------------------------------------------------------------------------------------------
def _shared_inputs(cfg, dist, seed, dtype):
    value, shapes, ref, off, logits = make_msda_inputs(cfg, dist, seed, dtype)
    off1, lg1 = off[:1].contiguous(), logits[:1].contiguous()
    rep = (value, shapes, ref, off1.expand_as(off).contiguous(), lg1.expand_as(logits).contiguous())
    return rep, (value, shapes, ref, off1, lg1)


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 2e-5), (torch.float16, 1e-3)])
@pytest.mark.parametrize("name,dist", [("tiny_sca", "G"), ("small_sca", "edge"), ("small_sca", "U")])
def test_shared_sca_matches_masked_camera_sum_of_oracle(name, dist, dtype, tol):
    from bevformer_tensorrt_b200.workloads import bev_reference_points_cam, camera_ring_lidar2img

    cfg = _cfg(name)
    rep, shared = _shared_inputs(cfg, dist, 103, dtype)
    if cfg.bev_hw[0] * cfg.bev_hw[1] == cfg.num_query:
        _, mask = bev_reference_points_cam(cfg.bev_hw, camera_ring_lidar2img(cfg.batch))
    else:
        mask = (torch.rand(cfg.batch, cfg.num_query, 1, generator=torch.Generator().manual_seed(3)) > 0.4).float()
        mask[:, :5] = 0  # queries no camera sees must come out as exact zeros (nothing pre-zeroes the output)
    per_cam = torch.from_numpy(_oracle_f32(rep))  # the plugin call with the repeated tensors
    want = (per_cam.reshape(cfg.batch, cfg.num_query, -1) * mask).sum(0)
    out = bt.multi_scale_deformable_attn_sca_shared(*_cuda(shared), mask.cuda())
    assert out.dtype == torch.float32 and out.shape == want.shape
    assert (out.cpu() - want).abs().max().item() < tol
    unseen = (mask.sum(0)[:, 0] == 0)
    assert unseen.any() and torch.equal(out.cpu()[unseen], torch.zeros_like(out.cpu()[unseen]))
    # and it is the same function as the per-camera fused op on the repeated tensors
    other = bt.multi_scale_deformable_attn_sca(*_cuda(rep), mask.cuda())
    assert (out - other).abs().max().item() < (2e-6 if dtype == torch.float32 else 2e-4)
    # offsets / logits with or without the leading singleton dimension
    out2 = bt.multi_scale_deformable_attn_sca_shared(*_cuda(shared[:3]), shared[3][0].cuda(), shared[4][0].cuda(),
                                                     mask.cuda())  # fmt: skip
    assert torch.equal(out2, out)


def test_shared_sca_base_shapes_and_errors():
    from bevformer_tensorrt_b200.workloads import bev_reference_points_cam, camera_ring_lidar2img

    cfg = CONFIGS["base_sca"]
    rep, shared = _shared_inputs(cfg, "G", 7, torch.float16)
    _, mask = bev_reference_points_cam(cfg.bev_hw, camera_ring_lidar2img(6))
    want = bt.multi_scale_deformable_attn_sca(*_cuda(rep), mask.cuda())
    n0 = _lib.launch_count()
    got = bt.multi_scale_deformable_attn_sca_shared(*_cuda(shared), mask.cuda())
    assert _lib.launch_count() == n0 + 1  # one kernel, no memset
    assert (got - want).abs().max().item() < 5e-4 and got.abs().max().item() > 0.1
    with pytest.raises(ValueError):  # the repeated tensors are not accepted silently
        bt.multi_scale_deformable_attn_sca_shared(*_cuda(rep), mask.cuda())
    with pytest.raises(RuntimeError):
        bt.multi_scale_deformable_attn_sca_shared(*shared, mask)


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-5), (torch.float16, FP16_TOL)])
def test_tsa_queue_mean_matches_mean_of_oracle(dtype, tol):
    """temporal_self_attention.py:447-453: plugin op on the 2-entry BEV queue, then mean over the queue."""
    cfg = _cfg("tsa_like")
    inputs = make_msda_inputs(cfg, "edge", 91, dtype)
    want = _oracle_f32(inputs).reshape(cfg.batch, cfg.num_query, -1).mean(0, keepdims=True)
    got = bt.multi_scale_deformable_attn_queue_mean(*_cuda(inputs))
    assert got.shape == (1, cfg.num_query, cfg.num_heads * cfg.channels) and got.dtype == dtype
    assert np.abs(got.float().cpu().numpy() - want).max() < tol


# ---------------------------------------------------------------------------------------------------------------
# host-buffer entry (bench.py's e2e leg): per-camera H2D / kernel / D2H pipeline
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_host_pipeline_equals_device_op(dtype):
    cfg = _cfg("small_sca")
    host = make_msda_inputs(cfg, "U", 5, dtype)
    want = bt.multi_scale_deformable_attn(*_cuda(host)).cpu()
    pinned = []
    for t in host:  # staging buffers from cudaHostAlloc (the recommended way), shapes stay a plain tensor
        if t.is_floating_point():
            h = bt.empty_pinned(t.shape, t.dtype)
            assert h.is_pinned() and h.shape == t.shape and h.dtype == t.dtype
            h.copy_(t)
            pinned.append(h)
        else:
            pinned.append(t)
    pipe = bt.HostMSDA(depth=2)  # fewer slots than cameras: slots are recycled inside one call
    out = pipe(*pinned)
    pipe.synchronize()
    assert out.is_pinned() and torch.equal(out, want)
    # back-to-back calls into the same output buffer, different inputs in between
    other = make_msda_inputs(cfg, "edge", 6, dtype)
    pinned2 = [t.pin_memory() if t.is_floating_point() else t for t in other]
    out2 = pipe(*pinned2)
    out3 = pipe(*pinned, out=torch.empty_like(out).pin_memory())
    pipe.synchronize()
    assert torch.equal(out2, bt.multi_scale_deformable_attn(*_cuda(other)).cpu()) and torch.equal(out3, want)
    with pytest.raises(RuntimeError):
        pipe(*_cuda(host))
