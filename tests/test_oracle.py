"""CPU suite, part 1: the oracle is pinned — against the committed golden vectors (produced by the
reference's own CPU kernels, tests/golden/gen_golden.py) and, when torchvision is importable here,
against the reference live on fresh seeds."""
import os

import numpy as np
import pytest


def test_nms_golden(oracle, golden):
    for i in range(3):
        keep = oracle.nms(golden[f"nms{i}_boxes"], golden[f"nms{i}_scores"], float(golden[f"nms{i}_thr"]), oracle.NMS_MODE_CPU)
        assert np.array_equal(keep, golden[f"nms{i}_keep"])
    keep = oracle.nms(golden["cfg1_boxes"], golden["cfg1_scores"], 0.5)
    assert np.array_equal(keep, golden["cfg1_keep"])


def test_nms_cuda_semantics_documented_difference(oracle):
    # SURVEY.md §2.2: the compiled CUDA reference contracts Sb into (Sa+Sb) and narrows the threshold.
    # a: area 3, b: area 3 — pick values where fma changes the last ulp is data dependent; here we only
    # require that both modes agree away from the threshold and are both greedy-consistent.
    rng = np.random.default_rng(0)
    b = rng.random((500, 4), dtype=np.float32) * 100
    b[:, 2:] += b[:, :2]
    s = rng.random(500, dtype=np.float32)
    k0, k1 = oracle.nms(b, s, 0.5, oracle.NMS_MODE_CPU), oracle.nms(b, s, 0.5, oracle.NMS_MODE_CUDA)
    assert np.array_equal(k0, k1)
    # threshold narrowing: iou == float(0.2) exactly is suppressed on CPU (0.2f > 0.2) but not on CUDA
    a = np.array([[0, 0, 10, 10], [0, 0, 10, 2]], dtype=np.float32)   # iou = 20/100 = 0.2f
    sc = np.array([1.0, 0.5], dtype=np.float32)
    assert list(oracle.nms(a, sc, 0.2, oracle.NMS_MODE_CPU)) == [0]
    assert list(oracle.nms(a, sc, 0.2, oracle.NMS_MODE_CUDA)) == [0, 1]


def test_nms_edge_cases(oracle):
    assert oracle.nms(np.zeros((0, 4), np.float32), np.zeros(0, np.float32), 0.5).size == 0
    one = oracle.nms(np.array([[0, 0, 1, 1]], np.float32), np.array([0.3], np.float32), 0.5)
    assert list(one) == [0]
    # ties keep index order (stable sort); identical boxes suppress each other
    b = np.tile(np.array([[0, 0, 4, 4]], np.float32), (5, 1))
    assert list(oracle.nms(b, np.ones(5, np.float32), 0.5)) == [0]
    # zero-area boxes: 0/0 = NaN > thr is False -> all kept
    z = np.tile(np.array([[1, 1, 1, 1]], np.float32), (3, 1))
    assert list(oracle.nms(z, np.array([3, 2, 1], np.float32), 0.5)) == [0, 1, 2]


def test_batched_nms_golden(oracle, golden):
    for name in ("bnms_trick", "bnms_vanilla"):
        b, s, i = golden[f"{name}_boxes"], golden[f"{name}_scores"], golden[f"{name}_idxs"]
        assert np.array_equal(oracle.batched_nms(b, s, i, 0.5), golden[f"{name}_keep"])
        assert np.array_equal(oracle.batched_nms(b, s, i, 0.5, strategy=1), golden[f"{name}_keep_v"])
        assert np.array_equal(oracle.batched_nms(b, s, i, 0.5, strategy=2), golden[f"{name}_keep_t"])


def test_roi_ops_golden(oracle, golden):
    x, rois = golden["roi_x"], golden["roi_rois"]
    for al in (0, 1):
        for sr in (2, -1):
            got = oracle.roi_align(x, rois, (7, 5), 0.25, sr, bool(al))
            assert np.array_equal(got, golden[f"roi_align_a{al}_s{sr}"])   # same arithmetic: bit-exact
    o, a = oracle.roi_pool(x, rois, (7, 5), 0.25)
    assert np.array_equal(o, golden["roi_pool_out"]) and np.array_equal(a, golden["roi_pool_argmax"])
    for sr in (2, -1):
        o, m = oracle.ps_roi_align(golden["psroi_x"], rois, (7, 5), 0.25, sr)
        np.testing.assert_array_equal(o, golden[f"psroi_s{sr}_out"])      # NaN == NaN position-wise
        assert np.array_equal(m, golden[f"psroi_s{sr}_map"])


def test_deform_conv2d_golden(oracle, golden):
    sh, sw, ph, pw, dh, dw = [int(v) for v in golden["dcn_args"]]
    for key, mask in (("dcn_out_mask", golden["dcn_mask"]), ("dcn_out_nomask", None)):
        got = oracle.deform_conv2d(golden["dcn_x"], golden["dcn_off"], golden["dcn_w"], golden["dcn_b"],
                                   (sh, sw), (ph, pw), (dh, dw), mask)
        np.testing.assert_allclose(got, golden[key], rtol=1e-5, atol=1e-5)
    empty = oracle.deform_conv2d(golden["dcn_x"][:0], golden["dcn_off"][:0], golden["dcn_w"], golden["dcn_b"],
                                 (sh, sw), (ph, pw), (dh, dw), None)
    assert empty.shape[0] == 0


def test_resize_golden(oracle, golden):
    img = golden["rs_img"]
    for mode, code in (("bilinear", 0), ("bicubic", 1)):
        for aa in (0, 1):
            for size in ((12, 13), (60, 80), (37, 20)):
                got = oracle.resize(img, size, code, bool(aa))
                np.testing.assert_allclose(got, golden[f"rs_{mode}_aa{aa}_{size[0]}x{size[1]}"], rtol=0, atol=1e-5)


# ---- live pin against the reference (importable in the build container) ------------------
tv = pytest.importorskip("torchvision", reason="reference wheel not importable: golden vectors still pin the oracle")


@pytest.mark.parametrize("seed", range(4))
@pytest.mark.parametrize("thr", [0.2, 0.5, 0.8])
def test_nms_live(oracle, seed, thr):
    import torch

    g = torch.Generator().manual_seed(seed)
    b = torch.rand(700, 4, generator=g) * 100
    b[:, 2:] += b[:, :2]
    s = torch.rand(700, generator=g)
    assert np.array_equal(tv.ops.nms(b, s, thr).numpy(), oracle.nms(b.numpy(), s.numpy(), thr))


def test_nms_float64_live(oracle):
    """The reference dispatches nms on float and double (cpu/nms_kernel.cpp:122-128); its own CUDA tests run
    in fp64 (test/test_ops.py:959-982)."""
    import torch

    g = torch.Generator().manual_seed(7)
    b = torch.rand(900, 4, generator=g, dtype=torch.float64) * 100
    b[:, 2:] += b[:, :2]
    s = torch.rand(900, generator=g, dtype=torch.float64)
    i = torch.randint(0, 6, (900,), generator=g)
    for thr in (0.2, 0.5, 0.8):
        assert np.array_equal(tv.ops.nms(b, s, thr).numpy(), oracle.nms(b.numpy(), s.numpy(), thr))
    assert np.array_equal(tv.ops.batched_nms(b, s, i, 0.5).numpy(), oracle.batched_nms(b.numpy(), s.numpy(), i.numpy(), 0.5))


def test_cfg3_batched_nms_live_reduced(oracle):
    """cfg3 at reduced size (20k boxes, 80 classes): reference vanilla path on CPU vs oracle."""
    import torch
    from vision_b200 import workloads

    b, s, i = workloads.cfg3_batched_nms(n=20_000)
    ref = tv.ops.batched_nms(b, s, i, 0.5).numpy()
    assert np.array_equal(ref, oracle.batched_nms(b.numpy(), s.numpy(), i.numpy(), 0.5))
    b, s, i = workloads.cfg3_batched_nms(n=20_000, clustered=True)
    ref = tv.ops.batched_nms(b, s, i, 0.5).numpy()
    assert np.array_equal(ref, oracle.batched_nms(b.numpy(), s.numpy(), i.numpy(), 0.5))


def test_cfg2_roi_align_live_reduced(oracle):
    import torch
    from vision_b200 import workloads

    x, rois, kw = workloads.cfg2_roi_align(channels=8, k=200)
    for aligned in (False, True):
        ref = tv.ops.roi_align(x, rois, kw["output_size"], kw["spatial_scale"], kw["sampling_ratio"], aligned).numpy()
        got = oracle.roi_align(x.numpy(), rois.numpy(), kw["output_size"], kw["spatial_scale"], kw["sampling_ratio"], aligned)
        assert np.array_equal(ref, got)


def test_resize_live_fp16_route(oracle):
    """_geometry.py:340-360: fp16 -> fp32 -> interpolate -> fp16."""
    import torch
    import torch.nn.functional as F

    x = torch.rand(1, 3, 270, 480).half()
    ref = F.interpolate(x.float(), size=[28, 28], mode="bilinear", align_corners=False, antialias=True).half()
    got = torch.from_numpy(oracle.resize(x.float().numpy(), (28, 28), 0, True)).half()
    assert (ref.float() - got.float()).abs().max().item() <= 1e-3


def test_extra_goldens_line_roi_align_fp64_nms_integer_resize(oracle, golden_extra):
    """tests/golden/reference_cpu_extra.npz (gen_golden_extra.py): the detection-head roi_align shape, float64 nms /
    batched_nms, and resize of uint8 / fp32 images routed as _geometry.py:340-360 routes CUDA tensors."""
    g = golden_extra
    for al in (0, 1):
        got = oracle.roi_align(g["line_x"], g["line_rois"], (7, 7), 0.25, 2, bool(al))
        assert np.array_equal(got, g[f"line_out_a{al}"])
    b, s, i = g["nms64_boxes"], g["nms64_scores"], g["nms64_idxs"]
    assert b.dtype == np.float64
    for k, thr in enumerate(g["nms64_thr"]):
        assert np.array_equal(oracle.nms(b, s, float(thr)), g[f"nms64_keep{k}"])
    assert np.array_equal(oracle.batched_nms(b, s, i, 0.5, strategy=1), g["bnms64_keep_v"])
    assert np.array_equal(oracle.batched_nms(b, s, i, 0.5, strategy=2), g["bnms64_keep_t"])
    for size in ((9, 20), (31, 200)):
        f = oracle.resize(g["rs8_img"].astype(np.float32), size, oracle.RESIZE_BILINEAR, True)
        want_f = g[f"rs8_float_{size[0]}x{size[1]}"]
        np.testing.assert_allclose(f, want_f, rtol=0, atol=2e-4)        # 0..255 scale
        out = np.rint(f).astype(np.uint8)                                 # round half to even, like Tensor.round_
        ties = np.abs(want_f - np.floor(want_f) - 0.5) < 1e-3
        assert np.array_equal(out[~ties], g[f"rs8_out_{size[0]}x{size[1]}"][~ties])
    np.testing.assert_allclose(oracle.resize(g["rsf_img"], (20, 60), oracle.RESIZE_BILINEAR, True), g["rsf_out_20x60"],
                               rtol=1e-6, atol=1e-6)


# ---- randomised live comparisons against the reference's CPU kernels (importable in the build container) ----
@pytest.mark.parametrize("seed", range(6))
def test_roi_ops_random_shapes_live(oracle, seed):
    """roi_align / roi_pool / ps_roi_align on random shapes, scales, pooled sizes and sampling ratios, RoIs partly
    outside the map: the oracle must reproduce the reference CPU kernels bit for bit (same arithmetic, same order)."""
    import torch

    g = torch.Generator().manual_seed(100 + seed)
    n_img, c = int(torch.randint(1, 4, (1,), generator=g)), int(torch.randint(1, 7, (1,), generator=g))
    h, w = int(torch.randint(5, 40, (1,), generator=g)), int(torch.randint(5, 40, (1,), generator=g))
    ph, pw = int(torch.randint(1, 8, (1,), generator=g)), int(torch.randint(1, 8, (1,), generator=g))
    scale = [1.0, 0.5, 0.25, 0.0625][seed % 4]
    sr = [-1, 1, 2, 3][(seed // 2) % 4]
    k = 17
    x = torch.randn(n_img, c, h, w, generator=g)
    r = torch.zeros(k, 5)
    r[:, 0] = torch.randint(0, n_img, (k,), generator=g).float()
    r[:, 1] = (torch.rand(k, generator=g) * 1.4 - 0.2) * w / scale
    r[:, 2] = (torch.rand(k, generator=g) * 1.4 - 0.2) * h / scale
    r[:, 3] = r[:, 1] + torch.rand(k, generator=g) * w / scale
    r[:, 4] = r[:, 2] + torch.rand(k, generator=g) * h / scale
    for aligned in (False, True):
        want = tv.ops.roi_align(x, r, (ph, pw), scale, sr, aligned).numpy()
        assert np.array_equal(oracle.roi_align(x.numpy(), r.numpy(), (ph, pw), scale, sr, aligned), want)
    po, pa = torch.ops.torchvision.roi_pool(x, r, scale, ph, pw)
    o, a = oracle.roi_pool(x.numpy(), r.numpy(), (ph, pw), scale)
    assert np.array_equal(o, po.numpy()) and np.array_equal(a, pa.numpy())
    xp = torch.randn(n_img, c * ph * pw, h, w, generator=g)
    o_ref, m_ref = torch.ops.torchvision.ps_roi_align(xp, r, scale, ph, pw, sr)
    o, m = oracle.ps_roi_align(xp.numpy(), r.numpy(), (ph, pw), scale, sr)
    assert np.array_equal(m, m_ref.numpy())
    np.testing.assert_array_equal(np.nan_to_num(o, nan=7.0, posinf=8.0, neginf=9.0),
                                  np.nan_to_num(o_ref.numpy(), nan=7.0, posinf=8.0, neginf=9.0))
    o_ref, m_ref = torch.ops.torchvision.ps_roi_pool(xp, r, scale, ph, pw)                 # cpu/ps_roi_pool_kernel.cpp
    o, m = oracle.ps_roi_pool(xp.numpy(), r.numpy(), (ph, pw), scale)
    assert np.array_equal(m, m_ref.numpy()) and np.array_equal(o, o_ref.numpy())


@pytest.mark.parametrize("seed", range(4))
def test_deform_conv2d_random_geometry_live(oracle, seed):
    import torch

    g = torch.Generator().manual_seed(200 + seed)
    groups, ogrps = [(1, 1), (2, 1), (1, 2), (2, 3)][seed]
    cin, cout = 6 * groups // groups * groups, 2 * groups
    cin = 6 if groups == 1 else 6
    cin = cin - cin % (groups * ogrps) + (groups * ogrps if cin % (groups * ogrps) else 0)
    kh, kw = [(3, 3), (1, 1), (3, 2), (2, 3)][seed]
    sh, sw = [(1, 1), (2, 2), (2, 1), (1, 2)][seed]
    ph, pw = [(1, 1), (0, 0), (1, 0), (2, 1)][seed]
    dh, dw = [(1, 1), (1, 1), (2, 1), (1, 2)][seed]
    b, ih, iw = 2, 9, 8
    oh = (ih + 2 * ph - (dh * (kh - 1) + 1)) // sh + 1
    ow = (iw + 2 * pw - (dw * (kw - 1) + 1)) // sw + 1
    x = torch.randn(b, cin, ih, iw, generator=g)
    off = torch.randn(b, ogrps * 2 * kh * kw, oh, ow, generator=g) * 1.5
    msk = torch.rand(b, ogrps * kh * kw, oh, ow, generator=g)
    wt = torch.randn(cout, cin // groups, kh, kw, generator=g)
    bias = torch.randn(cout, generator=g)
    for m in (msk, None):
        want = tv.ops.deform_conv2d(x, off, wt, bias, (sh, sw), (ph, pw), (dh, dw), m).numpy()
        got = oracle.deform_conv2d(x.numpy(), off.numpy(), wt.numpy(), bias.numpy(), (sh, sw), (ph, pw), (dh, dw),
                                   None if m is None else m.numpy())
        np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-5)     # the reference sums through a BLAS GEMM


@pytest.mark.parametrize("seed", range(4))
def test_resize_random_sizes_live(oracle, seed):
    import torch
    import torch.nn.functional as F

    g = torch.Generator().manual_seed(300 + seed)
    h, w = int(torch.randint(3, 90, (1,), generator=g)), int(torch.randint(3, 90, (1,), generator=g))
    oh, ow = int(torch.randint(1, 120, (1,), generator=g)), int(torch.randint(1, 120, (1,), generator=g))
    x = torch.rand(2, 2, h, w, generator=g)
    for mode, code in (("bilinear", oracle.RESIZE_BILINEAR), ("bicubic", oracle.RESIZE_BICUBIC)):
        for aa in (False, True):
            want = F.interpolate(x, size=[oh, ow], mode=mode, align_corners=False, antialias=aa).numpy()
            np.testing.assert_allclose(oracle.resize(x.numpy(), (oh, ow), code, aa), want, rtol=0, atol=5e-6)   # ATen vectorises the sums


# ---- box_iou_rotated: the oracle against the reference header itself (oracle/_ref) and the fixture made from it ----
def test_box_iou_rotated_golden_and_ref(oracle):
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "box_iou_rotated.npz"))
    assert np.array_equal(oracle.box_iou_rotated(g["boxes1"], g["boxes2"]), g["ious"])          # bit for bit
    u = oracle.box_iou_rotated(g["unit1"], g["unit2"])
    assert np.array_equal(u, g["unit_ious"])
    assert abs(u[0, 0] - 1.0) < 1e-6 and abs(u[0, 1] - 1.0 / 3.0) < 1e-6 and abs(u[0, 2] - 1.0) < 1e-6   # unit squares: 1, 1/3, 1 (90 degrees)
    rng = np.random.default_rng(7)
    c = rng.uniform(0, 100, (150, 2)); wh = np.exp(rng.uniform(0, 4, (150, 2))); a = rng.uniform(-360, 360, (150, 1))
    b = np.concatenate([c, wh, a], 1).astype(np.float32)
    assert np.array_equal(b, g["rand_boxes"])
    assert np.array_equal(oracle.box_iou_rotated(b, b[::-1].copy()), g["rand_ious"])    # the reference header's own result
    iou = oracle.box_iou_rotated(b, b)
    assert np.allclose(np.diag(iou), 1.0, atol=1e-5) and np.all(iou >= 0) and np.all(iou <= 1)
    np.testing.assert_allclose(iou, iou.T, atol=2e-5)       # symmetric up to the order of operations
