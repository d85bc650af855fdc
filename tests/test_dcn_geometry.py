"""deform_conv2d forward: every kernel against a plain fp64 reference, across the geometries each one accepts.

The forward has five kernels (tcgen05 16-bit, tcgen05 CTA pair, tcgen05 bf16x3 for fp32, SIMT, fp64) and the cfg4 tests
only reach the tensor-core ones at 3x3 / stride 1 / one offset group.  The cases below cover offset groups > 1 (the gather
groups' slab parity flips from one offset group to the next when the slab count is odd), 1x1 and rectangular kernels, stride,
padding and dilation, odd H*W (generic NHWC staging), output sizes that are not a multiple of 8 (scalar epilogue), ragged
pixel tiles, every tile width the 227 KB shared-memory limit admits, deep K on the fp32 kernel, and the SIMT kernel at sizes
with several M tiles and weight groups that straddle offset groups.

Each case asserts which kernel it reaches (workspace size and launch count), then runs twice:
  * dyadic data, where every path's arithmetic is exact: the output must equal the fp64 reference rounded to the dtype;
  * seeded randn data: max |err| / (atol + rtol |ref|) <= 1, 1e-5 for fp32 and 1e-2 for 16-bit storage.
"""
from __future__ import annotations

import os
from dataclasses import dataclass, field

import numpy as np
import pytest
import torch

DEV = "cuda"
_DT_CODE = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2, torch.float64: 3}
TOL = {torch.float32: (1e-5, 1e-5), torch.float16: (1e-2, 1e-2), torch.bfloat16: (1e-2, 1e-2), torch.float64: (1e-12, 1e-12)}


def _out_hw(h, w, kh, kw, stride, pad, dil):
    return ((h + 2 * pad[0] - (dil[0] * (kh - 1) + 1)) // stride[0] + 1,
            (w + 2 * pad[1] - (dil[1] * (kw - 1) + 1)) // stride[1] + 1)


# ---------------------------------------------------------------------------------------------------------------------
# fp64 reference
# ---------------------------------------------------------------------------------------------------------------------
def dcn_columns(x, off, stride, pad, dil, mask, kh, kw, offset_groups, pos_dtype=torch.float32):
    """Sampled columns [B, C_in, kh*kw, H_out*W_out] in fp64.  Sample positions are formed in `pos_dtype` (the op's own
    arithmetic type: fp32 for fp32 and for the 16-bit kernels, fp64 for fp64); everything after that is fp64, with the
    validity rules of bilinear_interpolate: y <= -1 or y >= H (x likewise) samples 0, each corner is checked on its own."""
    B, C, H, W = x.shape
    og = offset_groups
    ho, wo = _out_hw(H, W, kh, kw, stride, pad, dil)
    KK, HWo, cpo = kh * kw, ho * wo, C // og
    dev = x.device
    planes = x.double().reshape(B, og, cpo, H * W)
    offp = off.to(pos_dtype).reshape(B, og, KK, 2, HWo)
    mk = mask.double().reshape(B, og, KK, HWo) if mask is not None else None
    oy = torch.arange(ho, device=dev).repeat_interleave(wo)
    ox = torch.arange(wo, device=dev).repeat(ho)
    cols = torch.empty(B, og, cpo, KK, HWo, dtype=torch.float64, device=dev)
    for tap in range(KK):
        i, j = divmod(tap, kw)
        y = ((oy * stride[0] - pad[0] + i * dil[0]).to(pos_dtype) + offp[:, :, tap, 0]).double()    # [B, og, HWo]
        xx = ((ox * stride[1] - pad[1] + j * dil[1]).to(pos_dtype) + offp[:, :, tap, 1]).double()
        inside = ~((y <= -1) | (y >= H) | (xx <= -1) | (xx >= W))
        hl, wl = torch.floor(y), torch.floor(xx)
        lh, lw = y - hl, xx - wl
        hh, hw = 1 - lh, 1 - lw
        val = torch.zeros(B, og, cpo, HWo, dtype=torch.float64, device=dev)
        for cy, cx, wgt in ((hl, wl, hh * hw), (hl, wl + 1, hh * lw), (hl + 1, wl, lh * hw), (hl + 1, wl + 1, lh * lw)):
            ok = inside & (cy >= 0) & (cy <= H - 1) & (cx >= 0) & (cx <= W - 1)
            idx = (cy.clamp(0, H - 1) * W + cx.clamp(0, W - 1)).long()
            got = torch.gather(planes, 3, idx[:, :, None, :].expand(B, og, cpo, HWo))
            val += got * torch.where(ok, wgt, torch.zeros_like(wgt))[:, :, None, :]
        if mk is not None:
            val *= mk[:, :, tap][:, :, None, :]
        cols[:, :, :, tap] = val
    return cols.reshape(B, C, KK, HWo)


def dcn_ref(x, off, w, b, stride, pad, dil, mask, groups, offset_groups, pos_dtype=torch.float32, cols=None):
    """deform_conv2d in fp64 (plain torch; CPU or GPU): output [B, C_out, H_out, W_out]."""
    B, C, H, W = x.shape
    c_out, cin_g, kh, kw = w.shape
    ho, wo = _out_hw(H, W, kh, kw, stride, pad, dil)
    if cols is None:
        cols = dcn_columns(x, off, stride, pad, dil, mask, kh, kw, offset_groups, pos_dtype)
    cout_g = c_out // groups
    wd = w.double().reshape(groups, cout_g, cin_g * kh * kw)
    cg = cols.reshape(B, groups, cin_g * kh * kw, ho * wo)
    out = torch.einsum("gok,bgkp->bgop", wd, cg).reshape(B, c_out, ho, wo)
    if b is not None:
        out = out + b.double()[None, :, None, None]
    return out


def test_dcn_ref_matches_golden_reference_cpu(golden):
    """The reference CPU kernel's fp32 output on the test_ops.py geometry (og 3, groups 2, stride, dilation, kernel 3x2)."""
    g = golden
    sh, sw, ph, pw, dh, dw = [int(v) for v in g["dcn_args"]]
    x, off, w, b, m = (torch.from_numpy(g[k]) for k in ("dcn_x", "dcn_off", "dcn_w", "dcn_b", "dcn_mask"))
    og = off.shape[1] // (2 * w.shape[2] * w.shape[3])
    for key, mask in (("dcn_out_mask", m), ("dcn_out_nomask", None)):
        got = dcn_ref(x, off, w, b, (sh, sw), (ph, pw), (dh, dw), mask, x.shape[1] // w.shape[1], og)
        np.testing.assert_allclose(got.numpy(), g[key], rtol=1e-6, atol=1e-6)


# (C_in, C_out, (kh, kw), stride, pad, dil, groups, offset_groups, H, W, B, use_mask)
_TV_GEOMETRIES = [
    (6, 4, (3, 3), (1, 1), (1, 1), (1, 1), 1, 1, 7, 6, 2, True),
    (6, 4, (3, 2), (2, 1), (1, 0), (2, 1), 2, 3, 9, 8, 2, True),        # groups straddle offset groups
    (8, 6, (1, 1), (1, 1), (0, 0), (1, 1), 1, 4, 5, 7, 1, True),
    (12, 6, (2, 3), (1, 2), (0, 1), (1, 2), 3, 2, 8, 9, 2, False),      # 3 weight groups over 2 offset groups
    (4, 8, (5, 5), (2, 2), (2, 2), (1, 1), 2, 2, 11, 10, 1, True),
    (9, 3, (3, 1), (3, 1), (2, 0), (1, 3), 3, 1, 10, 5, 2, True),
    (10, 5, (2, 2), (1, 1), (3, 3), (2, 2), 5, 5, 6, 6, 3, True),
    (4, 4, (4, 3), (1, 1), (1, 1), (1, 1), 1, 2, 12, 4, 1, False),
]


def _edge_offsets(shape, h, w, g):
    """Offsets of randn*2, half of them replaced by multiples of 0.5 over [-(max(H,W)+3), max(H,W)+3]: many samples land
    exactly on -1, H-1, H (W likewise) and far outside."""
    span = max(h, w) + 3
    off = torch.randn(*shape, generator=g, dtype=torch.float64) * 2
    dy = torch.randint(-2 * span, 2 * span + 1, shape, generator=g).double() / 2
    return torch.where(torch.rand(*shape, generator=g) < 0.5, dy, off)


def test_dcn_ref_matches_torchvision_cpu_fp64():
    """With fp64 positions the reference equals the wheel's CPU deform_conv2d in fp64, including samples exactly on the
    -1 / H-1 / H borders and far outside."""
    tv = pytest.importorskip("torchvision")
    edges = 0
    for n, (cin, cout, (kh, kw), st, pd, dl, groups, og, h, w, bsz, use_mask) in enumerate(_TV_GEOMETRIES):
        g = torch.Generator().manual_seed(100 + n)
        ho, wo = _out_hw(h, w, kh, kw, st, pd, dl)
        x = torch.randn(bsz, cin, h, w, generator=g, dtype=torch.float64)
        wt = torch.randn(cout, cin // groups, kh, kw, generator=g, dtype=torch.float64)
        b = torch.randn(cout, generator=g, dtype=torch.float64)
        off = _edge_offsets((bsz, og * 2 * kh * kw, ho, wo), h, w, g)
        m = torch.rand(bsz, og * kh * kw, ho, wo, generator=g, dtype=torch.float64) if use_mask else None
        want = tv.ops.deform_conv2d(x, off, wt, b, st, pd, dl, m)
        got = dcn_ref(x, off, wt, b, st, pd, dl, m, groups, og, pos_dtype=torch.float64)
        np.testing.assert_allclose(got.numpy(), want.numpy(), rtol=1e-12, atol=1e-12, err_msg=f"geometry {n}")
        oy = torch.arange(ho).double()[:, None] * st[0] - pd[0]
        ys = torch.stack([oy + (t // kw) * dl[0] + off[:, 2 * (o * kh * kw + t)] for o in range(og) for t in range(kh * kw)])
        edges += int(((ys == -1) | (ys == h - 1) | (ys == h)).sum())
    assert edges > 100, edges          # the border rows were actually sampled


# ---------------------------------------------------------------------------------------------------------------------
# GPU cases
# ---------------------------------------------------------------------------------------------------------------------
BF16, FP16, FP32, FP64 = torch.bfloat16, torch.float16, torch.float32, torch.float64


@dataclass(frozen=True)
class Case:
    id: str
    dtypes: tuple
    cin: int
    cout: int
    k: tuple
    stride: tuple = (1, 1)
    pad: tuple = (0, 0)
    dil: tuple = (1, 1)
    og: int = 1
    groups: int = 1
    hw: tuple = (20, 20)
    batch: int = 2
    path: str = "tc"            # tc (deform_conv2d_tc[2]_kernel), tc3 (fp32 bf16x3), simt, f64
    bn: int = 0                 # tile width the tc path must pick (0: not a tc case)
    env: dict = field(default_factory=dict)
    mask: bool = True
    dyadic: bool = True


CASES = [
    # T1: 9 slabs per offset group (odd): the gather groups' slab parity flips at og 1
    Case("T1", (BF16, FP16), 128, 256, (3, 3), pad=(1, 1), og=2, bn=256),
    # T2: 1x1, one slab per og (one gather group idle in each og); odd H*W (generic NHWC staging); HWo 391: scalar epilogue
    Case("T2", (BF16, FP16), 256, 128, (1, 1), og=4, hw=(17, 23), bn=128, mask=False),
    # T3: BN 512 x 4 stages; stride / pad / dilation 2; HWo 17x24 = 408: vector epilogue + a ragged last tile
    Case("T3", (BF16, FP16), 64, 512, (3, 3), (2, 2), (2, 2), (2, 2), hw=(33, 47), bn=512),
    # T4: rectangular kernel, stride, pad and dilation; KK 15 (still BN 512 x 4 stages)
    Case("T4", (BF16,), 128, 512, (3, 5), (1, 2), (1, 2), (2, 1), og=2, hw=(24, 40), bn=512),
    # T5: 5x5 (KK 25): BN 512 and 256 do not fit, four N tiles of 128; with 3 stages BN 512 fits again (KK <= 26)
    Case("T5", (BF16, FP16), 64, 512, (5, 5), pad=(2, 2), bn=128),
    Case("T5-st3", (BF16, FP16), 64, 512, (5, 5), pad=(2, 2), bn=512, env={"VB200_DCN_STAGES": "3"}),
    # T6: HWo 81 < 128: one partial tile per image, three images
    Case("T6", (BF16,), 64, 128, (3, 3), pad=(1, 1), hw=(9, 9), batch=3, bn=128),
    Case("T7", (BF16, FP16), 128, 512, (3, 3), pad=(1, 1), og=2, bn=512),
    # F1: c_per_off 32 = one 32-channel slab per tap, 9 slabs per og (odd)
    Case("F1", (FP32,), 64, 128, (3, 3), (2, 2), (1, 1), og=2, hw=(31, 31), path="tc3"),
    Case("F2", (FP32,), 128, 256, (1, 1), og=4, hw=(17, 23), path="tc3", mask=False),
    # F3: KK 20, the largest the fp32 kernel's sampling table admits
    Case("F3", (FP32,), 64, 128, (4, 5), pad=(1, 2), hw=(24, 24), path="tc3"),
    # F4: K = 2048 x 9 on the fp32 kernel: accumulation bias at depth (randn only)
    Case("F4", (FP32,), 2048, 128, (3, 3), pad=(1, 1), hw=(12, 12), batch=1, path="tc3", dyadic=False),
    # S1: 7x7 (KK 49) fits no tensor-core tile
    Case("S1", (BF16, FP32), 64, 512, (7, 7), pad=(3, 3), hw=(24, 24), path="simt"),
    # S2: weight groups (24 channels) straddle offset groups (32 channels); cout_g 160 = two M tiles
    Case("S2", (FP16, FP32), 96, 640, (3, 3), pad=(1, 1), og=3, groups=4, path="simt"),
    # S3: c_out % 128 != 0
    Case("S3", (BF16,), 64, 96, (3, 3), pad=(1, 1), path="simt"),
    # D1: the fp64 kernel on the test_ops.py geometry, scaled up
    Case("D1", (FP64,), 24, 48, (3, 2), (2, 1), (1, 0), (2, 1), og=3, groups=2, hw=(19, 21), path="f64"),
]
# S4: every tensor-core shape again on the SIMT kernel (forced): SIMT at tensor-core depths of K
CASES += [Case("S4-" + c.id, c.dtypes if c.path == "tc3" else c.dtypes + (FP32,), c.cin, c.cout, c.k, c.stride, c.pad, c.dil, c.og,
               c.groups, c.hw, c.batch, "simt", 0, {**c.env, "VB200_DCN_PATH": "simt"}, c.mask, c.dyadic)
          for c in CASES if c.path in ("tc", "tc3") and not c.env]
BY_ID = {c.id: c for c in CASES}


class force_env:
    """Sets VB200_* overrides for the duration; the library reads them once, so each change goes through vb200_reload_env()
    (which also bumps the generation the packed-weight cache is keyed on)."""

    def __init__(self, env):
        self.env = dict(env)

    def __enter__(self):
        from vision_b200 import _lib

        self.old = {k: os.environ.get(k) for k in self.env}
        os.environ.update(self.env)
        _lib.core().vb200_reload_env()

    def __exit__(self, *a):
        from vision_b200 import _lib

        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        _lib.core().vb200_reload_env()


def _smem_optin():
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


def _tc_bn(cout, kk, env, smem):
    """tc_pick_bn() of deform_conv2d_tc.cu: the widest tile whose pipeline + [KK][128] sampling table fit `smem`."""
    st512 = 3 if env.get("VB200_DCN_STAGES") == "3" else 4

    def fits(bn):
        stages, kb = (3, 64) if bn <= 256 else (st512, 32)
        return stages * (128 + bn) * 2 * kb + 128 + kk * 128 * 32 + 1024 <= smem

    forced = env.get("VB200_DCN_BN")
    for bn in (512, 256, 128):
        if (forced is None or int(forced) == bn) and cout % bn == 0 and fits(bn):
            return bn
    return next((bn for bn in (512, 256, 128) if cout % bn == 0 and fits(bn)), 0)


def _make(case, dtype, dyadic, seed):
    """Inputs rounded to `dtype`.  Dyadic: x in {-2..2}, offsets k/2 in [-3, 3] (10 % at +-(max(H,W)+2)), mask in {0, .5, 1},
    weights in {+-.5, +-1} at a density that keeps >= 90 % of outputs below 16, bias k/2 -- every kernel's arithmetic is exact."""
    g = torch.Generator().manual_seed(seed)
    c, (h, w_) = case, case.hw
    kh, kw = c.k
    ho, wo = _out_hw(h, w_, kh, kw, c.stride, c.pad, c.dil)
    K = (c.cin // c.groups) * kh * kw
    xs, os_, ms = (c.batch, c.cin, h, w_), (c.batch, c.og * 2 * kh * kw, ho, wo), (c.batch, c.og * kh * kw, ho, wo)
    ws = (c.cout, c.cin // c.groups, kh, kw)
    if dyadic:
        x = torch.randint(-2, 3, xs, generator=g).double()
        off = torch.randint(-6, 7, os_, generator=g).double() / 2
        far = torch.rand(os_, generator=g) < 0.1
        off = torch.where(far, (max(h, w_) + 2) * torch.sign(torch.rand(os_, generator=g) - 0.5).double(), off)
        m = torch.randint(0, 3, ms, generator=g).double() / 2
        density = min(0.2, 64.0 / K)
        mag = torch.randint(1, 3, ws, generator=g).double() / 2 * torch.sign(torch.rand(ws, generator=g) - 0.5).double()
        wt = torch.where(torch.rand(ws, generator=g) < density, mag, torch.zeros_like(mag))
        b = torch.randint(-4, 5, (c.cout,), generator=g).double() / 2
    else:
        x = torch.randn(xs, generator=g, dtype=torch.float64)
        off = torch.randn(os_, generator=g, dtype=torch.float64) * 2
        m = torch.rand(ms, generator=g, dtype=torch.float64)
        wt = torch.randn(ws, generator=g, dtype=torch.float64) / K ** 0.5
        b = torch.randn(c.cout, generator=g, dtype=torch.float64)
    cast = lambda t: t.to(dtype).to(DEV)
    return cast(x), cast(off), cast(wt), cast(b), (cast(m) if c.mask else None)


def _run(vb, case, dtype, data, env=None):
    """One call on a fresh weight, with the routing asserted: workspace > 0 exactly on the tensor-core paths, and the launch
    count of a first call (weight pack + NCHW->NHWC staging + main kernel = 3 on a tensor-core path; 1 otherwise)."""
    from vision_b200 import _lib

    x, off, w, b, m = data
    env = {**case.env, **(env or {})}
    kh, kw = case.k
    ho, wo = _out_hw(*case.hw, kh, kw, case.stride, case.pad, case.dil)
    with force_env(env):
        wsb = _lib.core().vb200_deform_conv2d_workspace_bytes(_DT_CODE[dtype], case.batch, case.cin, case.hw[0], case.hw[1], case.cout,
                                                              kh, kw, ho, wo, case.groups, case.og)
        before = vb.launch_count()
        got = vb.ops.deform_conv2d(x, off, w, b, case.stride, case.pad, case.dil, m)
        launches = vb.launch_count() - before
    tensor_core = case.path in ("tc", "tc3")
    assert (wsb > 0) == tensor_core, (case.id, wsb)
    assert launches == (3 if tensor_core else 1), (case.id, launches)
    if case.path == "tc":
        assert _tc_bn(case.cout, kh * kw, env, _smem_optin()) == case.bn, "the case no longer reaches the tile it is meant to test"
    assert got.dtype == dtype and got.shape == (case.batch, case.cout, ho, wo)
    return got


def _ref(case, data, dtype):
    x, off, w, b, m = data
    kh, kw = case.k
    pos = torch.float64 if dtype == torch.float64 else torch.float32
    cols = dcn_columns(x, off, case.stride, case.pad, case.dil, m, kh, kw, case.og, pos)
    ref = dcn_ref(x, off, w, b, case.stride, case.pad, case.dil, m, case.groups, case.og, cols=cols)
    return ref, cols


def _assert_exact(case, data, dtype, got, ref, cols):
    x, off, w, b, m = data
    # bit budget: every partial sum is a multiple of 1/16 below 2^16, so fp32 accumulation in any order is exact
    bound = dcn_ref(x, off, w.abs(), b.abs(), case.stride, case.pad, case.dil, m, case.groups, case.og, cols=cols.abs())
    assert bound.max().item() * 16 < 2 ** 20, bound.max().item()
    small = (ref.abs() < 16).double().mean().item()
    assert small >= 0.9, small           # one wrong term (+-1/16) changes the stored bits, even in bf16
    want = ref.to(dtype)
    if not torch.equal(got, want):
        bad = (got != want).nonzero()
        i = tuple(bad[0].tolist())
        raise AssertionError(f"{case.id} {dtype}: {bad.shape[0]} of {got.numel()} outputs differ; first at {i}: "
                             f"got {got[i].item()} want {want[i].item()}")


def _worst(got, ref, dtype):
    atol, rtol = TOL[dtype]
    return ((got.double() - ref).abs() / (atol + rtol * ref.abs())).max().item()


def _params(dyadic):
    return [pytest.param(c, dt, id=f"{c.id}-{str(dt).split('.')[-1]}") for c in CASES for dt in c.dtypes if c.dyadic or not dyadic]


@pytest.mark.gpu
@pytest.mark.parametrize("case,dtype", _params(dyadic=True))
def test_dcn_exact_on_dyadic_data(vb, case, dtype):
    data = _make(case, dtype, dyadic=True, seed=sum(map(ord, case.id)))
    got = _run(vb, case, dtype, data)
    ref, cols = _ref(case, data, dtype)
    _assert_exact(case, data, dtype, got, ref, cols)


@pytest.mark.gpu
@pytest.mark.parametrize("case,dtype", _params(dyadic=False))
def test_dcn_randn_within_tolerance(vb, case, dtype):
    data = _make(case, dtype, dyadic=False, seed=7)
    got = _run(vb, case, dtype, data)
    ref, _ = _ref(case, data, dtype)
    worst = _worst(got, ref, dtype)
    atol, rtol = TOL[dtype]
    assert worst <= 1, f"{case.id} {dtype}: max |err| / ({atol} + {rtol} |ref|) = {worst:.3f}"


_T7_VARIANTS = [{"VB200_DCN_BN": "128"}, {"VB200_DCN_BN": "256"}, {"VB200_DCN_BN": "512"},
                {"VB200_DCN_STAGES": "3"}, {"VB200_DCN_STAGES": "4"},
                {"VB200_DCN_BLEND": "16"}, {"VB200_DCN_BLEND": "32"}, {"VB200_DCN_CTA2": "1"}]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [BF16, FP16])
def test_dcn_forced_variants_match_default_bit_for_bit(vb, dtype):
    """Every tile width, pipeline depth, blend and the CTA-pair kernel on one og-2 shape: the same bits as the default path
    (and as the reference) on dyadic data."""
    case = BY_ID["T7"]
    data = _make(case, dtype, dyadic=True, seed=17)
    ref, cols = _ref(case, data, dtype)
    default = _run(vb, case, dtype, data)
    _assert_exact(case, data, dtype, default, ref, cols)
    smem = _smem_optin()
    for env in _T7_VARIANTS:
        if "VB200_DCN_BN" in env:
            assert _tc_bn(case.cout, 9, env, smem) == int(env["VB200_DCN_BN"]), env      # the forced tile fits: it is really used
        variant = Case(**{**case.__dict__, "env": env, "bn": _tc_bn(case.cout, 9, env, smem)})
        got = _run(vb, variant, dtype, data)
        assert torch.equal(got, default), env


@pytest.mark.gpu
@pytest.mark.parametrize("case_id,dtype", [("T2", BF16), ("T2", FP16), ("T4", BF16)])
def test_dcn_packed_weight_and_channels_last_beyond_cfg4(vb, case_id, dtype):
    """Second call with the same weight: no pack launch; channels-last input: no staging launch either; same bits."""
    case = BY_ID[case_id]
    x, off, w, b, m = _make(case, dtype, dyadic=False, seed=23)
    xcl = x.contiguous(memory_format=torch.channels_last)
    outs, launches = [], []
    for inp in (x, x, xcl):
        before = vb.launch_count()
        outs.append(vb.ops.deform_conv2d(inp, off, w, b, case.stride, case.pad, case.dil, m))
        launches.append(vb.launch_count() - before)
    assert launches == [3, 2, 1]           # pack + staging + kernel; kernel + staging; kernel
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])


@pytest.mark.gpu
@pytest.mark.parametrize("case_id,dtype", [("T2", BF16), ("T3", BF16), ("T3", FP16)])
def test_dcn_gather_destinations_beyond_cfg4(vb, case_id, dtype):
    """deform_conv2d_gather from the scalar (T2) and the transposing vector (T3) epilogue: each of three destinations equals
    the plain op and the guard elements around each are untouched."""
    case = BY_ID[case_id]
    x, off, w, b, m = _make(case, dtype, dyadic=False, seed=29)
    mm = m if m is not None else torch.zeros(case.batch, 1, device=DEV, dtype=dtype)
    geo = (*case.stride, *case.pad, *case.dil, case.groups, case.og, m is not None)
    want = torch.ops.vision_b200.deform_conv2d(x, w, off, mm, b, *geo)
    n = want.numel()
    bufs = [torch.full((n + 128,), 5.0, dtype=dtype, device=DEV) for _ in range(3)]
    ptrs = [t.data_ptr() + 64 * t.element_size() for t in bufs]
    torch.ops.vision_b200.deform_conv2d_gather(x, w, off, mm, b, ptrs, *geo)
    for t in bufs:
        assert torch.equal(t[64:64 + n].view(want.shape), want)
        assert bool((t[:64] == 5).all()) and bool((t[64 + n:] == 5).all())
