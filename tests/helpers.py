"""Shared test helpers (tests may use oracle/; the product package may not)."""
import glob
import hashlib
import os

import numpy as np
import torch

from bevformer_tensorrt_b200.workloads import MSDAConfig, make_msda_inputs

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def input_digest(*tensors):
    h = hashlib.sha256()
    for t in tensors:
        h.update(t.contiguous().numpy().tobytes())
    return h.hexdigest()


def sample_index(numel, k, seed=0):
    """Sorted flat indices of a fixed, seeded sample of about k elements of an output with numel elements (the form in
    which tests/golden stores outputs too large for a fixture)."""
    return np.unique(np.random.default_rng(seed).integers(0, numel, k))


def load_ref_kernels(name):
    """Outputs of the reference's own CUDA kernels (tests/golden/make_golden_ref_kernels.py)."""
    return np.load(os.path.join(GOLDEN, f"ref_kernels_{name}.npz"))


def check_digest(z, key, *tensors):
    assert input_digest(*tensors) == str(z[f"{key}_digest"]), f"{key}: the seeded inputs no longer match the fixture"


def golden_msda_cases():
    return sorted(glob.glob(os.path.join(GOLDEN, "msda_*.npz")))


def load_golden_msda(path):
    """Returns (cfg, (value, shapes, ref, off, logits) float32 CPU tensors, expected out ndarray)."""
    z = np.load(path)
    B, Q, M, C, L, P, G, seed = (int(x) for x in z["meta"])
    shapes = tuple((int(h), int(w)) for h, w in z["shapes"])
    cfg = MSDAConfig(os.path.basename(path), B, Q, M, C, shapes, P, G)
    inputs = make_msda_inputs(cfg, str(z["dist"]), seed, torch.float32)
    if input_digest(*inputs) != str(z["digest"]):
        if "value" in z.files:  # self-contained fixture
            inputs = (torch.from_numpy(z["value"]), inputs[1], torch.from_numpy(z["ref"]),
                      torch.from_numpy(z["off"]), torch.from_numpy(z["logits"]))  # fmt: skip
        else:
            raise RuntimeError(f"{path}: seeded CPU generator no longer reproduces the golden inputs")
    return cfg, inputs, z["out"]


def make_grid_sampler_inputs(N, C, Hi, Wi, Ho, Wo, seed=0, depth=None, span=15.0):
    """input ~ N(0,1); grid = a regular sweep over [-span, span] (1.5x beyond the image, as the reference test's
    linspace(-15, 15), test_grid_sampler.py:29-36) plus N(0, 0.5) jitter, channel-first [N, 2|3, ...]."""
    g = torch.Generator().manual_seed(seed)
    if depth is None:
        inp = torch.randn(N, C, Hi, Wi, generator=g)
        ys, xs = torch.meshgrid(torch.linspace(-span, span, Ho), torch.linspace(-span, span, Wo), indexing="ij")
        grid = torch.stack([xs, ys], 0)[None].repeat(N, 1, 1, 1)
    else:
        Di, Do = depth
        inp = torch.randn(N, C, Di, Hi, Wi, generator=g)
        zs, ys, xs = torch.meshgrid(torch.linspace(-span, span, Do), torch.linspace(-span, span, Ho),
                                    torch.linspace(-span, span, Wo), indexing="ij")  # fmt: skip
        grid = torch.stack([xs, ys, zs], 0)[None].repeat(N, 1, 1, 1, 1)
    grid = grid + 0.5 * torch.randn(grid.shape, generator=g)
    return inp, grid.contiguous()


def make_rotation_grid(H, W, angle_deg, shift=(0.0, 0.0)):
    """The prev-BEV warp grid of BASELINE configs[3]: output pixel centres rotated by ``angle_deg`` about the image
    centre (plus a translation in pixels), normalised to [-1, 1] and scaled x10 — the plugin's [-10, 10] convention
    (SURVEY.md Appendix B; onnx_ops.py:226-232 builds the same grid x10). Returns float32 [1, 2, H, W] (x plane, y)."""
    import math

    ys, xs = torch.meshgrid(torch.arange(H, dtype=torch.float32), torch.arange(W, dtype=torch.float32), indexing="ij")
    cx, cy = (W - 1) / 2.0, (H - 1) / 2.0
    c, s_ = math.cos(math.radians(angle_deg)), math.sin(math.radians(angle_deg))
    sx = c * (xs - cx) - s_ * (ys - cy) + cx + shift[0]
    sy = s_ * (xs - cx) + c * (ys - cy) + cy + shift[1]
    gx = ((sx + 0.5) / W * 2 - 1) * 10
    gy = ((sy + 0.5) / H * 2 - 1) * 10
    return torch.stack([gx, gy], 0)[None].contiguous()


ROTATE_CASES = {
    # name: (C, H, W, angle_deg, (center_x, center_y))
    "bev_small": (8, 50, 50, 1.7, (25.0, 25.0)),        # prev_bev alignment: a few degrees about the BEV centre
    "bev_neg": (6, 40, 48, -4.25, (24.0, 20.0)),
    "big_angle": (5, 33, 47, 127.3, (20.5, 13.25)),     # reference test: angle ~ N(0,1)*360 (test_rotate.py:21-25)
    "off_center": (4, 31, 29, -61.0, (40.0, 38.0)),     # centre outside the image (test_rotate.py: center = 500, 500)
    "zero": (3, 17, 19, 0.0, (9.5, 8.5)),
    "right_angle": (3, 16, 16, 90.0, (8.0, 8.0)),       # lands on x.5 / integer source indices
    "odd_c": (7, 21, 23, 33.3, (11.0, 10.0)),           # C not a multiple of the kCHW2 / kCHW4 packet
}


def make_rotate_inputs(case, seed=0):
    """img ~ N(0,1) [C,H,W], angle [1] (degrees), center [2] as float32 tensors (test_rotate.py:19-26)."""
    C, H, W, ang, ctr = ROTATE_CASES[case]
    g = torch.Generator().manual_seed(seed)
    return torch.randn(C, H, W, generator=g), torch.tensor([ang]), torch.tensor(list(ctr))


_PC_RANGE = (-51.2, -51.2, -5.0, 51.2, 51.2, 3.0)  # BEVFormer nuScenes configs (point_cloud_range)
POINT_SAMPLING_CASES = {
    # name: (bev_h, bev_w, num_points_in_pillar, image (h, w), pc_range)
    "ring_small": (50, 50, 4, (928, 1600), _PC_RANGE),     # BEVFormer-tiny BEV size
    "ring_rect": (30, 44, 4, (480, 800), _PC_RANGE),       # non-square BEV, small images (BEVFormer-small-like)
    "ring_d8": (20, 20, 8, (928, 1600), (-40.0, -40.0, -1.0, 40.0, 40.0, 5.4)),
    "ring_d1": (16, 24, 1, (928, 1600), _PC_RANGE),
}


def make_point_sampling_inputs(case):
    """lidar2img [6, 4, 4] float32 of the synthetic camera ring (bevformer_tensorrt_b200.workloads)."""
    from bevformer_tensorrt_b200.workloads import camera_ring_lidar2img

    return camera_ring_lidar2img(6, img_hw=POINT_SAMPLING_CASES[case][3])


DCN_CASES = {
    # name: (N, Ci, H, W, Co, kh, kw, stride, padding, dilation, groups, deform_groups)
    "k3_s1_p1_g2_dg2": (2, 16, 13, 17, 12, 3, 3, 1, 1, 1, 2, 2),  # the reference op test's structure, reduced
    "k3_s2_p1_g1_dg1": (2, 8, 14, 15, 6, 3, 3, 2, 1, 1, 1, 1),
    "k3_s1_p2_d2_g1_dg4": (1, 16, 12, 12, 8, 3, 3, 1, 2, 2, 1, 4),
    "k1_s1_p0_g1_dg1": (2, 8, 9, 9, 8, 1, 1, 1, 0, 1, 1, 1),
    "k3x5_s1_p1_g1_dg1": (1, 4, 11, 13, 4, 3, 5, 1, 1, 1, 1, 1),
    "backbone_like": (2, 64, 29, 50, 64, 3, 3, 1, 1, 1, 1, 1),  # BEVFormer R101 stage shapes, channels reduced
    # shapes the fused tcgen05 path takes in FP16 (groups = dg = 1, C % 64 == 0, Co in {128, 256, 512})
    "fused_co128": (2, 64, 20, 24, 128, 3, 3, 1, 1, 1, 1, 1),
    "fused_co256_ragged": (3, 128, 29, 50, 256, 3, 3, 1, 1, 1, 1, 1),  # 1450 pixels: partial last tile, unaligned rows
    "fused_co512_s2": (1, 64, 31, 33, 512, 3, 3, 2, 1, 1, 1, 1),
    "fused_k1": (2, 128, 16, 16, 128, 1, 1, 1, 0, 1, 1, 1),
}


def make_dcn_inputs(case, seed=0, dtype=torch.float32):
    N, Ci, H, W, Co, kh, kw, s, p, d, g, dg = DCN_CASES[case]
    gen = torch.Generator().manual_seed(seed)
    Ho = (H + 2 * p - (d * (kh - 1) + 1)) // s + 1
    Wo = (W + 2 * p - (d * (kw - 1) + 1)) // s + 1
    x = torch.randn(N, Ci, H, W, generator=gen)
    off = torch.randn(N, dg * 2 * kh * kw, Ho, Wo, generator=gen) * 1.5
    mask = torch.sigmoid(torch.randn(N, dg * kh * kw, Ho, Wo, generator=gen))  # dcn.py:74
    w = torch.randn(Co, Ci // g, kh, kw, generator=gen) / (Ci // g * kh * kw) ** 0.5
    b = torch.randn(Co, generator=gen)
    kwargs = dict(stride=s, padding=p, dilation=d, groups=g, deform_groups=dg)
    if torch.__version__ and kh != kw:
        pass
    return x.to(dtype), off.to(dtype), mask.to(dtype), w.to(dtype), b.to(dtype), kwargs
