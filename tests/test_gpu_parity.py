"""GPU suite (-m gpu): the CUDA kernels, called through the C ABI (via the torch shim, and once
directly through ctypes), against (a) the committed golden vectors of the reference CPU kernels,
(b) the CPU oracle on seeded inputs — at BASELINE.json sizes where the oracle finishes in seconds,
(c) size-independent properties, (d) the reference's CUDA kernels on the same box when the
torchvision wheel is importable (an extra; never required).

Tolerances (BASELINE.json north_star): bit-exact kept indices for nms / batched_nms; 1e-5 for fp32
roi_align / roi_pool / ps_roi_align / resize / deform_conv2d; 1e-2 for 16-bit storage types."""
import ctypes
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

F32_TOL = dict(rtol=1e-5, atol=1e-5)
F16_TOL = dict(rtol=1e-2, atol=1e-2)
DEV = "cuda"


def t(a, dtype=None):
    x = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return x if dtype is None else x.to(dtype)


def npy(x):
    return x.detach().float().cpu().numpy() if x.is_floating_point() else x.detach().cpu().numpy()


class force_env:
    def __init__(self, key, val):
        self.key, self.val = key, val

    def __enter__(self):
        from vision_b200 import _lib

        self.old = os.environ.get(self.key)
        os.environ[self.key] = self.val
        _lib.core().vb200_reload_env()          # the library reads its overrides once, not per call

    def __exit__(self, *a):
        from vision_b200 import _lib

        if self.old is None:
            os.environ.pop(self.key, None)
        else:
            os.environ[self.key] = self.old
        _lib.core().vb200_reload_env()


def test_native_library_loaded(vb):
    """The process must have the in-tree .so mapped — no eager / library fallback."""
    maps = open("/proc/self/maps").read()
    assert "libvision_b200.so" in maps and "libvision_b200_torch.so" in maps
    assert torch.ops.vision_b200._abi_version() == 1


# =============================== roi_align ===================================
@pytest.mark.parametrize("aligned", [0, 1])
@pytest.mark.parametrize("sr", [2, -1])
def test_roi_align_golden(vb, golden, aligned, sr):
    x, rois = t(golden["roi_x"]), t(golden["roi_rois"])
    want = golden[f"roi_align_a{aligned}_s{sr}"]
    before = vb.launch_count()
    got = vb.ops.roi_align(x, rois, (7, 5), 0.25, sr, bool(aligned))
    assert vb.launch_count() > before, "no vision_b200 kernel was launched"
    np.testing.assert_allclose(npy(got), want, **F32_TOL)
    # the generic kernel restates the reference CPU arithmetic op for op: expect bit equality
    assert np.array_equal(npy(got), want)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64, torch.float16])
@pytest.mark.parametrize("contiguous", [True, False])
def test_roi_align_reference_test_shapes(vb, oracle, dtype, contiguous):
    # test/test_ops.py:127-163 (RoIOpTester.test_forward): x = rand(2, 50, 10, 10), 4 fixed RoIs, pool 5x5
    torch.manual_seed(0)
    x = torch.rand(2, 50, 10, 10, dtype=dtype, device=DEV)
    if not contiguous:
        x = x.permute(0, 1, 3, 2)
    rois = torch.tensor([[0, 0, 0, 9, 9], [0, 0, 5, 4, 9], [0, 5, 5, 9, 9], [1, 0, 0, 9, 9]], dtype=dtype, device=DEV)
    for aligned in (False, True):
        got = vb.ops.roi_align(x, rois, 5, spatial_scale=1, sampling_ratio=-1, aligned=aligned)
        want = oracle.roi_align(npy(x), npy(rois), 5, 1.0, -1, aligned)
        tol = F16_TOL if dtype == torch.float16 else F32_TOL
        np.testing.assert_allclose(npy(got), want, **tol)
        assert got.dtype == dtype and got.shape == (4, 50, 5, 5)


@pytest.mark.parametrize("aligned", [False, True])
def test_roi_align_cfg2_full_size_vs_oracle(vb, oracle, aligned):
    """BASELINE configs[1] at full size: 1x256x200x272 fp32, 1000 RoIs, 7x7, sr=2 (plane-resident kernel)."""
    from vision_b200 import workloads

    x, rois, kw = workloads.cfg2_roi_align()
    want = oracle.roi_align(x.numpy(), rois.numpy(), kw["output_size"], kw["spatial_scale"], kw["sampling_ratio"], aligned)
    got = vb.ops.roi_align(x.to(DEV), rois.to(DEV), kw["output_size"], kw["spatial_scale"], kw["sampling_ratio"], aligned)
    np.testing.assert_allclose(npy(got), want, **F32_TOL)
    with force_env("VB200_ROI_ALIGN_PATH", "generic"):
        got_g = vb.ops.roi_align(x.to(DEV), rois.to(DEV), kw["output_size"], kw["spatial_scale"], kw["sampling_ratio"], aligned)
    assert np.array_equal(npy(got_g), want)


def test_roi_align_plane_path_batched_and_sampling_ratios(vb, oracle):
    from vision_b200 import workloads

    for sr in (1, 3, 4):
        x, rois, kw = workloads.cfg2_roi_align(seed=sr, k=300, batch=3, channels=7, height=40, width=52)
        with force_env("VB200_ROI_ALIGN_PATH", "plane"):
            got = vb.ops.roi_align(x.to(DEV), rois.to(DEV), (3, 6), 0.25, sr, True)
        want = oracle.roi_align(x.numpy(), rois.numpy(), (3, 6), 0.25, sr, True)
        np.testing.assert_allclose(npy(got), want, **F32_TOL)


def test_roi_align_line_path(vb, oracle):
    """7x7 / sampling_ratio 2 takes the line-wise kernel: batched maps, odd widths, RoIs hanging outside the
    map (zero rows / zero columns), degenerate and border-hugging RoIs, both lane orientations."""
    from vision_b200 import workloads

    # k = 2500 exceeds the sorted-table limit (caller's order, no load overlap); the others use sorted tables
    for seed, (b, c, h, w), k in ((1, (3, 7, 40, 53), 300), (2, (1, 24, 64, 31), 257), (3, (2, 5, 33, 200), 500),
                                  (4, (1, 3, 50, 60), 2500), (5, (1, 300, 20, 24), 40)):
        x, rois, kw = workloads.cfg2_roi_align(seed=seed, k=k, batch=b, channels=c, height=h, width=w)
        rois = rois.clone()
        rois[::7, 1:3] -= 90.0                      # start outside the map
        rois[1::11, 3:] += 400.0                    # end far outside
        rois[2::13, 3:] = rois[2::13, 1:3]          # zero-size
        rois[3::17, 1:] = torch.tensor([w * 4 - 6.0, h * 4 - 6.0, w * 4 + 0.0, h * 4 + 0.0])   # bottom-right corner
        rois[4::19, 3] = rois[4::19, 1] + 700.0     # very wide, short
        for aligned in (False, True):
            want = oracle.roi_align(x.numpy(), rois.numpy(), 7, 0.25, 2, aligned)
            with force_env("VB200_ROI_ALIGN_PATH", "line"):
                got = vb.ops.roi_align(x.to(DEV), rois.to(DEV), 7, 0.25, 2, aligned)
            np.testing.assert_allclose(npy(got), want, **F32_TOL)
            with force_env("VB200_ROI_ALIGN_PATH", "plane"):
                if w % 4 == 0:
                    got = vb.ops.roi_align(x.to(DEV), rois.to(DEV), 7, 0.25, 2, aligned)
                    np.testing.assert_allclose(npy(got), want, **F32_TOL)


def test_roi_align_band_path(vb, oracle):
    """7x7 / sampling_ratio 2 / channels % 8 == 0 takes the band-resident channel-interleaved kernel: several bands per
    map (bin rows straddling two bands are summed with RED into rows the geometry kernel zeroed), batched maps, RoIs
    hanging outside the map, degenerate / inverted / border-hugging RoIs, out-of-range batch indices (zeros)."""
    from vision_b200 import workloads

    for seed, (b, c, h, w), k in ((1, (2, 8, 80, 200), 300), (2, (1, 16, 200, 272), 200), (3, (1, 8, 300, 100), 400),
                                  (4, (3, 24, 40, 53), 500), (5, (1, 64, 33, 31), 70)):
        x, rois, kw = workloads.cfg2_roi_align(seed=seed, k=k, batch=b, channels=c, height=h, width=w)
        rois = rois.clone()
        rois[::7, 1:3] -= 90.0                      # start outside the map
        rois[1::11, 3:] += 400.0                    # end far outside
        rois[2::13, 3:] = rois[2::13, 1:3]          # zero-size
        rois[3::17, 1:] = torch.tensor([w * 4 - 6.0, h * 4 - 6.0, w * 4 + 0.0, h * 4 + 0.0])   # bottom-right corner
        rois[4::19, 3] = rois[4::19, 1] + 700.0     # very wide, short
        rois[5::23, 4] = rois[5::23, 2] + 2000.0    # taller than the map
        rois[6::29, 2] = h * 4 + 50.0               # entirely below the map: every sample row is outside
        rois[6::29, 4] = h * 4 + 90.0
        rois[8::31, 3:] = rois[8::31, 1:3] - 40.0   # inverted (aligned=True keeps the negative size)
        for aligned in (False, True):
            want = oracle.roi_align(x.numpy(), rois.numpy(), 7, 0.25, 2, aligned)
            with force_env("VB200_ROI_ALIGN_PATH", "band"):
                before = vb.launch_count()
                got = vb.ops.roi_align(x.to(DEV), rois.to(DEV), 7, 0.25, 2, aligned)
                assert vb.launch_count() - before == 2      # geometry + gather
                again = vb.ops.roi_align(x.to(DEV), rois.to(DEV), 7, 0.25, 2, aligned)
            np.testing.assert_allclose(npy(got), want, **F32_TOL)
            assert torch.equal(got, again), "band kernel must be bit-reproducible (split bin rows add two partials)"
    # batch indices outside [0, B): zeros, like the line kernel
    x, rois, kw = workloads.cfg2_roi_align(seed=9, k=64, batch=2, channels=8, height=60, width=80)
    rois[::5, 0] = 7.0
    rois[1::5, 0] = -1.0
    with force_env("VB200_ROI_ALIGN_PATH", "band"):
        got = vb.ops.roi_align(x.to(DEV), rois.to(DEV), 7, 0.25, 2, False)
    ok = (rois[:, 0] >= 0) & (rois[:, 0] < 2)
    want = oracle.roi_align(x.numpy(), rois[ok].numpy(), 7, 0.25, 2, False)
    np.testing.assert_allclose(npy(got)[ok.numpy()], want, **F32_TOL)
    assert float(got[~ok.to(DEV)].abs().max()) == 0.0


def test_roi_align_cfg2_thread_per_bin_plane_path(vb, oracle):
    from vision_b200 import workloads

    x, rois, kw = workloads.cfg2_roi_align(channels=16)
    want = oracle.roi_align(x.numpy(), rois.numpy(), 7, 0.25, 2, False)
    with force_env("VB200_ROI_ALIGN_PATH", "plane"):
        got = vb.ops.roi_align(x.to(DEV), rois.to(DEV), 7, 0.25, 2, False)
    np.testing.assert_allclose(npy(got), want, **F32_TOL)


def test_roi_align_edge_cases(vb, oracle):
    x = torch.randn(1, 3, 8, 8, device=DEV)
    assert vb.ops.roi_align(x, torch.zeros(0, 5, device=DEV), 7).shape == (0, 3, 7, 7)
    # list-of-boxes input, boxes hanging outside the map, huge adaptive grid (table overflow path)
    boxes = [torch.tensor([[-20.0, -20.0, 30.0, 30.0], [2.0, 2.0, 2.0, 2.0]], device=DEV)]
    got = vb.ops.roi_align(x, boxes, 2, 1.0, -1, False)
    rois = np.array([[0, -20, -20, 30, 30], [0, 2, 2, 2, 2]], np.float32)
    np.testing.assert_allclose(npy(got), oracle.roi_align(npy(x), rois, 2, 1.0, -1, False), **F32_TOL)
    big = torch.randn(1, 2, 600, 600, device=DEV)
    r = torch.tensor([[0, 0.0, 0.0, 599.0, 599.0]], device=DEV)
    got = vb.ops.roi_align(big, r, 1, 1.0, -1, False)     # grid 599x599 > table capacity
    np.testing.assert_allclose(npy(got), oracle.roi_align(npy(big), npy(r), 1, 1.0, -1, False), rtol=1e-4, atol=1e-4)
    with pytest.raises(RuntimeError, match="Tensor\\[K, 5\\]"):
        torch.ops.vision_b200.roi_align(x, torch.zeros(2, 4, device=DEV), 1.0, 2, 2, 2, False)
    with pytest.raises(RuntimeError, match="same type"):
        torch.ops.vision_b200.roi_align(x, torch.zeros(2, 5, device=DEV, dtype=torch.float64), 1.0, 2, 2, 2, False)


# =============================== roi_pool / ps_roi_align =======================
def test_roi_pool_golden_and_random(vb, oracle, golden):
    out, arg = torch.ops.vision_b200.roi_pool(t(golden["roi_x"]), t(golden["roi_rois"]), 0.25, 7, 5)
    assert np.array_equal(npy(out), golden["roi_pool_out"]) and np.array_equal(npy(arg), golden["roi_pool_argmax"])
    from vision_b200 import workloads

    x, rois, kw = workloads.cfg2_roi_align(channels=16, k=200)
    o, a = torch.ops.vision_b200.roi_pool(x.to(DEV), rois.to(DEV), 0.25, 7, 7)
    wo, wa = oracle.roi_pool(x.numpy(), rois.numpy(), 7, 0.25)
    assert np.array_equal(npy(o), wo) and np.array_equal(npy(a), wa)            # bit-exact incl. argmax
    # fp16: the reference kernel runs its box arithmetic in Half (every scalar op rounds to half), which moves some bin
    # windows; our kernel reproduces those roundings, so the check is bit-equality with the reference's own CUDA kernel
    xh = x.half().to(DEV)
    oh, ah = torch.ops.vision_b200.roi_pool(xh, rois.half().to(DEV), 0.25, 7, 7)
    tv = pytest.importorskip("torchvision")
    assert not vb.installed()
    rh_, rah = torch.ops.torchvision.roi_pool(xh, rois.half().to(DEV), 0.25, 7, 7)
    assert torch.equal(oh, rh_) and torch.equal(ah, rah)


def test_ps_roi_align_golden_and_random(vb, oracle, golden):
    for sr in (2, -1):
        out, mp = torch.ops.vision_b200.ps_roi_align(t(golden["psroi_x"]), t(golden["roi_rois"]), 0.25, 7, 5, sr)
        np.testing.assert_array_equal(npy(out), golden[f"psroi_s{sr}_out"])     # incl. NaN/inf of degenerate RoIs
        assert np.array_equal(npy(mp), golden[f"psroi_s{sr}_map"])
    torch.manual_seed(1)
    x = torch.randn(2, 5 * 49, 30, 41)
    rois = torch.tensor([[0, 4.0, 4.0, 100.0, 90.0], [1, 10.0, 20.0, 150.0, 110.0], [1, 0.0, 0.0, 163.0, 119.0]])
    got = vb.ops.ps_roi_align(x.to(DEV), rois.to(DEV), 7, 0.25, 2)
    want, _ = oracle.ps_roi_align(x.numpy(), rois.numpy(), 7, 0.25, 2)
    np.testing.assert_allclose(npy(got), want, **F32_TOL)
    with pytest.raises(RuntimeError, match="multiple of pooling height"):
        vb.ops.ps_roi_align(torch.randn(1, 50, 8, 8, device=DEV), rois[:1].to(DEV), 7, 1.0, 2)


# =============================== nms ==========================================
def _set(vb, which):
    vb.set_nms_semantics(which)


def test_nms_golden_cpu_semantics(vb, golden):
    _set(vb, "cpu")
    try:
        for i in range(3):
            keep = vb.ops.nms(t(golden[f"nms{i}_boxes"]), t(golden[f"nms{i}_scores"]), float(golden[f"nms{i}_thr"]))
            assert keep.dtype == torch.int64 and np.array_equal(npy(keep), golden[f"nms{i}_keep"])
        keep = vb.ops.nms(t(golden["cfg1_boxes"]), t(golden["cfg1_scores"]), 0.5)
        assert np.array_equal(npy(keep), golden["cfg1_keep"])
    finally:
        _set(vb, "cuda")


@pytest.mark.parametrize("n", [1, 2, 63, 64, 65, 129, 1000, 3072, 3073, 9000])
@pytest.mark.parametrize("sem", ["cpu", "cuda"])
def test_nms_vs_oracle_sizes(vb, oracle, n, sem):
    """Covers the one-CTA segment kernel (n <= 3072) and the tiled mask + scan path (n > 3072)."""
    rng = np.random.default_rng(n)
    b = (rng.random((n, 4), dtype=np.float32) * 100)
    b[:, 2:] = b[:, :2] + rng.random((n, 2), dtype=np.float32) * 30 + 0.5
    s = rng.random(n, dtype=np.float32)
    s[::7] = s[0]                                  # ties: stable order decides
    _set(vb, sem)
    try:
        for thr in (0.3, 0.5, 0.7):
            keep = vb.ops.nms(t(b), t(s), thr)
            want = oracle.nms(b, s, thr, oracle.NMS_MODE_CPU if sem == "cpu" else oracle.NMS_MODE_CUDA)
            assert np.array_equal(npy(keep), want), (n, sem, thr)
    finally:
        _set(vb, "cuda")


@pytest.mark.parametrize("sem", ["cpu", "cuda"])
def test_nms_float64(vb, oracle, sem):
    """fp64 boxes (test/test_ops.py:959-982 compares CPU and CUDA nms in fp64): segment kernel, mask path, batched."""
    rng = np.random.default_rng(11)
    mode = oracle.NMS_MODE_CPU if sem == "cpu" else oracle.NMS_MODE_CUDA
    _set(vb, sem)
    try:
        for n in (500, 5000):
            b = rng.random((n, 4)) * 100
            b[:, 2:] = b[:, :2] + rng.random((n, 2)) * 30 + 0.5
            s = rng.random(n)
            keep = vb.ops.nms(t(b), t(s), 0.5)
            assert keep.dtype == torch.int64 and np.array_equal(npy(keep), oracle.nms(b, s, 0.5, mode))
        n = 40_000
        b = rng.random((n, 4)) * 300
        b[:, 2:] = b[:, :2] + rng.random((n, 2)) * 60 + 1
        s = rng.permutation(n).astype(np.float64) / n
        i = rng.integers(0, 20, n)
        keep = vb.ops.batched_nms(t(b), t(s), t(i), 0.5)
        assert np.array_equal(npy(keep), oracle.batched_nms(b, s, i, 0.5, mode=mode, device_is_cuda=True))
    finally:
        _set(vb, "cuda")
    tv = pytest.importorskip("torchvision")
    assert torch.equal(tv.ops.nms(t(b[:3000]), t(s[:3000]), 0.5), vb.ops.nms(t(b[:3000]), t(s[:3000]), 0.5))


@pytest.mark.parametrize("path", ["chain", "mask"])
def test_nms_both_suppression_paths(vb, oracle, path):
    """Plain nms: the single-CTA sequential kernel and the all-SM IoU mask + scan give the oracle's indices at
    sizes either side of the switch-over, in both arithmetics and for fp64."""
    rng = np.random.default_rng(23)
    for n in (1, 63, 64, 65, 300, 2500, 5000):
        b = rng.random((n, 4), dtype=np.float32) * 100
        b[:, 2:] = b[:, :2] + rng.random((n, 2), dtype=np.float32) * 40 + 0.5
        s = rng.random(n, dtype=np.float32)
        for sem, mode in (("cuda", oracle.NMS_MODE_CUDA), ("cpu", oracle.NMS_MODE_CPU)):
            _set(vb, sem)
            try:
                with force_env("VB200_NMS_PATH", path):
                    keep = vb.ops.nms(t(b), t(s), 0.3)
                    keep64 = vb.ops.nms(t(b.astype(np.float64)), t(s.astype(np.float64)), 0.3) if n in (65, 2500) else None
            finally:
                _set(vb, "cuda")
            assert np.array_equal(npy(keep), oracle.nms(b, s, 0.3, mode)), (n, sem, path)
            if keep64 is not None:
                assert np.array_equal(npy(keep64), oracle.nms(b.astype(np.float64), s.astype(np.float64), 0.3, mode))
    # degenerate boxes (zero area, inverted) push the mask kernel onto its exact-only branch
    n = 700
    b = rng.random((n, 4), dtype=np.float32) * 50
    b[:, 2:] = b[:, :2] + rng.random((n, 2), dtype=np.float32) * 30
    b[::5, 2] = b[::5, 0]                      # zero width
    b[3::11, [0, 2]] = b[3::11, [2, 0]]        # inverted
    s = rng.random(n, dtype=np.float32)
    with force_env("VB200_NMS_PATH", path):
        keep = vb.ops.nms(t(b), t(s), 0.4)
    assert np.array_equal(npy(keep), oracle.nms(b, s, 0.4, oracle.NMS_MODE_CUDA))


def test_nms_threshold_narrowing_semantics(vb):
    a = torch.tensor([[0, 0, 10, 10], [0, 0, 10, 2]], dtype=torch.float32, device=DEV)   # iou == 0.2f exactly
    sc = torch.tensor([1.0, 0.5], device=DEV)
    _set(vb, "cpu")
    assert vb.ops.nms(a, sc, 0.2).tolist() == [0]
    _set(vb, "cuda")
    assert vb.ops.nms(a, sc, 0.2).tolist() == [0, 1]


def test_nms_edge_cases_and_errors(vb):
    assert vb.ops.nms(torch.zeros(0, 4, device=DEV), torch.zeros(0, device=DEV), 0.5).shape == (0,)
    z = torch.ones(3, 4, device=DEV)                                    # zero-area boxes: NaN > thr is False
    assert vb.ops.nms(z, torch.tensor([3.0, 2.0, 1.0], device=DEV), 0.5).tolist() == [0, 1, 2]
    same = torch.tensor([[0, 0, 4, 4.0]] * 5, device=DEV)
    assert vb.ops.nms(same, torch.ones(5, device=DEV), 0.5).tolist() == [0]
    # test/test_ops.py:927-935
    for bad in ((torch.rand(4, device=DEV), torch.rand(3, device=DEV)), (torch.rand(3, 5, device=DEV), torch.rand(3, device=DEV)),
                (torch.rand(3, 4, device=DEV), torch.rand(3, 2, device=DEV)), (torch.rand(3, 4, device=DEV), torch.rand(4, device=DEV))):
        with pytest.raises(RuntimeError):
            vb.ops.nms(bad[0], bad[1], 0.5)
    # fp16 literal boxes of test_nms_float16 (test/test_ops.py:1010-1017)
    boxes = torch.tensor([[285.3538, 185.5758, 1193.5110, 851.4551], [285.1472, 188.7374, 1192.4984, 851.0669],
                          [279.2440, 197.9812, 1189.4746, 849.2019]], device=DEV)
    scores = torch.tensor([0.6370, 0.7569, 0.3966], device=DEV)
    assert torch.equal(vb.ops.nms(boxes, scores, 0.2), vb.ops.nms(boxes.half(), scores.half(), 0.2))


# =============================== batched_nms ===================================
def test_batched_nms_golden(vb, golden):
    _set(vb, "cpu")
    try:
        g = golden
        keep = vb.ops.batched_nms(t(g["bnms_trick_boxes"]), t(g["bnms_trick_scores"]), t(g["bnms_trick_idxs"]), 0.5)
        assert np.array_equal(npy(keep), g["bnms_trick_keep_t"])          # numel 2400 <= 100k on CUDA -> trick
        keep = vb.ops.batched_nms(t(g["bnms_vanilla_boxes"]), t(g["bnms_vanilla_scores"]), t(g["bnms_vanilla_idxs"]), 0.5)
        assert np.array_equal(npy(keep), g["bnms_vanilla_keep_t"])        # numel 12000 <= 100k on CUDA -> trick
    finally:
        _set(vb, "cuda")


@pytest.mark.parametrize("clustered", [False, True])
@pytest.mark.parametrize("sem", ["cpu", "cuda"])
def test_batched_nms_cfg3_full_size_vs_oracle(vb, oracle, clustered, sem):
    """BASELINE configs[2] at full size: 100k boxes x 80 classes (vanilla semantics, numel 400k > 100k)."""
    from vision_b200 import workloads

    b, s, i = workloads.cfg3_batched_nms(clustered=clustered)
    mode = oracle.NMS_MODE_CPU if sem == "cpu" else oracle.NMS_MODE_CUDA
    want = oracle.batched_nms(b.numpy(), s.numpy(), i.numpy(), 0.5, mode=mode, device_is_cuda=True)
    _set(vb, sem)
    try:
        before = vb.launch_count()
        keep = vb.ops.batched_nms(b.to(DEV), s.to(DEV), i.to(DEV), 0.5)
        assert vb.launch_count() > before
    finally:
        _set(vb, "cuda")
    assert keep.dtype == torch.int64 and np.array_equal(npy(keep), want)
    # properties: unique indices, scores non-increasing, per-class greedy validity is implied by equality
    k = npy(keep)
    assert len(np.unique(k)) == len(k) and np.all(np.diff(s.numpy()[k]) <= 0)


def test_batched_nms_strategies_classes_and_edges(vb, oracle):
    rng = np.random.default_rng(5)
    for n, ncls, ids in ((3000, 4, None), (30_000, 3, None), (26_000, 1, None), (26_000, 26_000, None), (27_000, 5, "weird")):
        b = rng.random((n, 4), dtype=np.float32) * 200
        b[:, 2:] = b[:, :2] + rng.random((n, 2), dtype=np.float32) * 60 + 1
        s = (rng.permutation(n).astype(np.float32)) / n
        i = rng.integers(0, ncls, n).astype(np.int64)
        if ids == "weird":
            i = np.array([-7, 0, 3, 2**40, -2**35], dtype=np.int64)[i]     # arbitrary int64 class ids
        keep = vb.ops.batched_nms(t(b), t(s), t(i), 0.5)
        want = oracle.batched_nms(b, s, i, 0.5, mode=oracle.NMS_MODE_CUDA, device_is_cuda=True)
        assert np.array_equal(npy(keep), want), (n, ncls, ids)
    e = vb.ops.batched_nms(torch.zeros(0, 4, device=DEV), torch.zeros(0, device=DEV), torch.zeros(0, dtype=torch.int64, device=DEV), 0.5)
    assert e.shape == (0,) and e.dtype == torch.int64


def test_batched_nms_mask_scan_and_chain_paths_agree(vb, oracle):
    """Classes of <= 2048 boxes go through the all-SM IoU mask + bit-word scan, longer ones through the per-class
    sequential chain, in the same call; VB200_BNMS_PATH=chain pins the sequential kernel."""
    rng = np.random.default_rng(17)
    n = 40_000
    b = rng.random((n, 4), dtype=np.float32) * 300
    b[:, 2:] = b[:, :2] + rng.random((n, 2), dtype=np.float32) * 80 + 1
    s = (rng.permutation(n).astype(np.float32)) / n
    i = rng.integers(1, 40, n).astype(np.int64)
    i[:6000] = 0                       # one class of 6000+ boxes (sequential path), 39 of ~870 (mask path)
    i[6000:6003] = 77                  # a 3-box class
    i[6003] = 78                       # a single-box class
    for sem, mode in (("cuda", oracle.NMS_MODE_CUDA), ("cpu", oracle.NMS_MODE_CPU)):
        want = oracle.batched_nms(b, s, i, 0.4, mode=mode, device_is_cuda=True)
        _set(vb, sem)
        try:
            keep = vb.ops.batched_nms(t(b), t(s), t(i), 0.4)
            with force_env("VB200_BNMS_PATH", "chain"):
                keep_chain = vb.ops.batched_nms(t(b), t(s), t(i), 0.4)
        finally:
            _set(vb, "cuda")
        assert np.array_equal(npy(keep), want) and np.array_equal(npy(keep_chain), want)
    # segment boundaries on and around 64-position block edges, class sizes 63/64/65/128/2048/2049
    sizes = [63, 64, 65, 128, 1, 2048, 2049, 191] + [700] * 35      # n > 25000: vanilla semantics
    i = np.repeat(np.arange(len(sizes)), sizes).astype(np.int64)
    n = len(i)
    b = rng.random((n, 4), dtype=np.float32) * 120
    b[:, 2:] = b[:, :2] + rng.random((n, 2), dtype=np.float32) * 50 + 1
    s = (rng.permutation(n).astype(np.float32)) / n
    perm = rng.permutation(n)
    b, s, i = b[perm], s[perm], i[perm]
    keep = vb.ops.batched_nms(t(b), t(s), t(i), 0.5)
    assert np.array_equal(npy(keep), oracle.batched_nms(b, s, i, 0.5, mode=oracle.NMS_MODE_CUDA, device_is_cuda=True))


# =============================== deform_conv2d ==================================
def test_deform_conv2d_golden(vb, golden):
    g = golden
    sh, sw, ph, pw, dh, dw = [int(v) for v in g["dcn_args"]]
    for key, mask in (("dcn_out_mask", t(g["dcn_mask"])), ("dcn_out_nomask", None)):
        got = vb.ops.deform_conv2d(t(g["dcn_x"]), t(g["dcn_off"]), t(g["dcn_w"]), t(g["dcn_b"]), (sh, sw), (ph, pw), (dh, dw), mask)
        np.testing.assert_allclose(npy(got), g[key], **F32_TOL)


@pytest.mark.parametrize("batch", [0, 33])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
def test_deform_conv2d_reference_test_geometry(vb, oracle, batch, dtype):
    # test/test_ops.py:1113-1167 get_fn_args: groups 2, offset groups 3, stride (2,1), pad (1,0), dil (2,1), kernel (3,2)
    torch.manual_seed(0)
    cin, cout, g, og, sh, sw, ph, pw, dh, dw, kh, kw, ih, iw = 6, 2, 2, 3, 2, 1, 1, 0, 2, 1, 3, 2, 5, 4
    oh = (ih + 2 * ph - (dh * (kh - 1) + 1)) // sh + 1
    ow = (iw + 2 * pw - (dw * (kw - 1) + 1)) // sw + 1
    x = torch.rand(batch, cin, ih, iw).to(dtype)
    off = torch.randn(batch, og * 2 * kh * kw, oh, ow).to(dtype)
    msk = torch.randn(batch, og * kh * kw, oh, ow).to(dtype)
    w = torch.randn(cout, cin // g, kh, kw).to(dtype)
    bias = torch.randn(cout).to(dtype)
    for mask in (msk, None):
        got = vb.ops.deform_conv2d(x.to(DEV), off.to(DEV), w.to(DEV), bias.to(DEV), (sh, sw), (ph, pw), (dh, dw),
                                   None if mask is None else mask.to(DEV))
        assert got.shape == (batch, cout, oh, ow) and got.dtype == dtype
        if batch:
            want = oracle.deform_conv2d(x.float().numpy(), off.float().numpy(), w.float().numpy(), bias.float().numpy(),
                                        (sh, sw), (ph, pw), (dh, dw), None if mask is None else mask.float().numpy())
            np.testing.assert_allclose(npy(got), want, **(F32_TOL if dtype == torch.float32 else dict(rtol=1e-2, atol=1e-2)))   # north_star: 1e-2 for 16-bit
    # non-contiguous inputs are accepted (reference calls .contiguous())
    if batch:
        xt = x.to(DEV).permute(0, 1, 3, 2).contiguous().permute(0, 1, 3, 2)
        a = vb.ops.deform_conv2d(xt, off.to(DEV), w.to(DEV), bias.to(DEV), (sh, sw), (ph, pw), (dh, dw), msk.to(DEV))
        b = vb.ops.deform_conv2d(x.to(DEV), off.to(DEV), w.to(DEV), bias.to(DEV), (sh, sw), (ph, pw), (dh, dw), msk.to(DEV))
        assert torch.equal(a, b)


def test_deform_conv2d_errors(vb):
    x = torch.rand(1, 6, 5, 4, device=DEV)
    w = torch.rand(2, 3, 3, 2, device=DEV)
    off = torch.rand(1, 3 * 2 * 6, 2, 3, device=DEV)
    with pytest.raises(RuntimeError, match="mask.shape\\[1\\] is not valid"):
        vb.ops.deform_conv2d(x, off, w, None, (2, 1), (1, 0), (2, 1), torch.rand(1, 5, 2, 3, device=DEV))
    with pytest.raises(RuntimeError, match="the shape of the offset tensor"):
        vb.ops.deform_conv2d(x, torch.rand(1, 2, 2, 3, device=DEV), w, None, (2, 1), (1, 0), (2, 1))
    with pytest.raises(RuntimeError, match="offset.shape\\[1\\] is not valid"):
        vb.ops.deform_conv2d(x, torch.rand(1, 3 * 2 * 6 + 12, 2, 3, device=DEV)[:, :3 * 2 * 6 + 1], w, None, (2, 1), (1, 0), (2, 1))


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-5), (torch.bfloat16, 1e-2), (torch.float16, 1e-2)])
def test_deform_conv2d_cfg4_reduced_vs_oracle(vb, oracle, dtype, tol):
    """cfg4 geometry (3x3, stride 1, pad 1, DCNv2) at N=2, C 64->128, 32x32: inputs rounded to `dtype`,
    reference arithmetic in fp32 on the rounded values (the reference has no bf16 kernel)."""
    from vision_b200 import workloads

    x, off, w, b, m = workloads.cfg4_deform_conv2d(batch=2, c_in=64, c_out=128, hw=32, dtype=dtype)
    if dtype != torch.float32:
        # one accumulator (BN 128/256, 3 stages) and two accumulators (BN 512, 4 stages) of the tcgen05 kernel
        for c_out, hw in ((256, 16), (512, 12)):
            x2, off2, w2, b2, m2 = workloads.cfg4_deform_conv2d(seed=c_out, batch=1, c_in=128, c_out=c_out, hw=hw, dtype=dtype)
            want2 = oracle.deform_conv2d(x2.float().numpy(), off2.float().numpy(), w2.float().numpy(), b2.float().numpy(),
                                         (1, 1), (1, 1), (1, 1), m2.float().numpy())
            got2 = vb.ops.deform_conv2d(x2.to(DEV), off2.to(DEV), w2.to(DEV), b2.to(DEV), 1, 1, 1, m2.to(DEV))
            np.testing.assert_allclose(npy(got2), want2, rtol=tol, atol=tol)
    want = oracle.deform_conv2d(x.float().numpy(), off.float().numpy(), w.float().numpy(), b.float().numpy(), (1, 1), (1, 1), (1, 1),
                                m.float().numpy())
    got = vb.ops.deform_conv2d(x.to(DEV), off.to(DEV), w.to(DEV), b.to(DEV), 1, 1, 1, m.to(DEV))
    np.testing.assert_allclose(npy(got), want, rtol=tol, atol=tol)


def test_deform_conv2d_cta_pair_variant_matches(vb, oracle):
    """The cta_group::2 (CTA-pair, M = 256) tcgen05 kernel, enabled by VB200_DCN_CTA2=1: same bits as the
    single-CTA kernel, incl. an odd tile count (padded cluster) and ragged pixel tiles; oracle parity."""
    from vision_b200 import workloads

    for batch, cin, cout, hw in ((1, 64, 512, 12), (3, 128, 512, 20)):
        x, off, w, b, m = workloads.cfg4_deform_conv2d(seed=hw, batch=batch, c_in=cin, c_out=cout, hw=hw, dtype=torch.bfloat16)
        args = (x.to(DEV), off.to(DEV), w.to(DEV), b.to(DEV), 1, 1, 1, m.to(DEV))
        one = vb.ops.deform_conv2d(*args)
        with force_env("VB200_DCN_CTA2", "1"):
            two = vb.ops.deform_conv2d(*args)
        assert torch.equal(one, two)
        want = oracle.deform_conv2d(x.float().numpy(), off.float().numpy(), w.float().numpy(), b.float().numpy(), (1, 1), (1, 1), (1, 1),
                                    m.float().numpy())
        np.testing.assert_allclose(npy(two), want, rtol=1e-2, atol=1e-2)


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-5), (torch.bfloat16, 1e-2)])
def test_deform_conv2d_zero_offset_is_conv2d(vb, dtype, tol):
    """Property at a larger size: offsets 0 and no mask == plain convolution (fp64 convolution of the same rounded values
    as the ground truth, so the bound is on OUR error only: 1e-5 fp32 / 1e-2 bf16 as north_star states)."""
    from vision_b200 import workloads

    x, off, w, b, _ = workloads.cfg4_deform_conv2d(batch=4, c_in=256, c_out=256, hw=64, dtype=dtype, offset_scale=0.0, use_mask=False)
    x, off, w, b = x.to(DEV), off.to(DEV), w.to(DEV), b.to(DEV)
    got = vb.ops.deform_conv2d(x, off, w, b, 1, 1, 1, None)
    want = torch.nn.functional.conv2d(x.double(), w.double(), b.double(), stride=1, padding=1)
    np.testing.assert_allclose(got.double().cpu().numpy(), want.cpu().numpy(), rtol=tol, atol=tol)


# =============================== resize =========================================
@pytest.mark.parametrize("mode", ["bilinear", "bicubic"])
@pytest.mark.parametrize("aa", [0, 1])
def test_resize_golden(vb, golden, mode, aa):
    img = t(golden["rs_img"])
    for size in ((12, 13), (60, 80), (37, 20)):
        got = vb.transforms.resize_image(img, list(size), interpolation=mode, antialias=bool(aa))
        np.testing.assert_allclose(npy(got), golden[f"rs_{mode}_aa{aa}_{size[0]}x{size[1]}"], rtol=0, atol=1e-5)


@pytest.mark.parametrize("aa", [True, False])
def test_resize_cfg5_reduced_batch_vs_oracle(vb, oracle, aa):
    """cfg5 geometry at batch 2: 2x3x2160x3840 fp16 -> 224x224 (reference route: fp16->fp32->interp->fp16)."""
    from vision_b200 import workloads

    x = workloads.cfg5_resize(device=DEV, batch=2)
    got = vb.transforms.resize(x, [224, 224], antialias=aa)
    assert got.shape == (2, 3, 224, 224) and got.dtype == torch.float16
    want = torch.from_numpy(oracle.resize(x.float().cpu().numpy(), (224, 224), 0, aa)).half().float().numpy()
    np.testing.assert_allclose(npy(got), want, rtol=1e-2, atol=1e-3)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float32, torch.uint8])
@pytest.mark.parametrize("shape,size", [((3, 2, 96, 1024), (17, 40)), ((5, 301, 1000), (33, 97)), ((1, 1, 64, 4000), (64, 160)),
                                        ((2, 3, 500, 808), (224, 224)), ((2, 400, 1600), (7, 3))])
def test_resize_stream_path_vs_generic_and_oracle(vb, oracle, dtype, shape, size):
    """The streaming bilinear-AA downscale kernel (scale_w >= 2, 16-bit storage) against the generic
    kernel and the oracle: pixel-pair slot widths LW 4/6/10/16, band splitting, ragged last intervals."""
    torch.manual_seed(sum(shape))
    if dtype == torch.uint8:
        x = torch.randint(0, 256, shape, dtype=torch.uint8).to(DEV)
    else:
        x = torch.randn(*shape).to(dtype).to(DEV)
    fast = vb.transforms.resize_image(x.unsqueeze(-3) if x.dim() == 2 else x, list(size), antialias=True)
    with force_env("VB200_RESIZE_PATH", "generic"):
        slow = vb.transforms.resize_image(x, list(size), antialias=True)
    assert fast.dtype == dtype and fast.shape == slow.shape
    want = oracle.resize(x.float().cpu().numpy(), size, 0, True)
    if dtype == torch.uint8:
        # _geometry.py:352-359: round (half to even) then cast; the two kernels sum in different orders, so a value
        # within 1e-4 of a .5 tie may round differently
        f, s_ = npy(fast).astype(np.float32), npy(slow).astype(np.float32)
        assert np.abs(f - np.rint(want)).max() <= 1.0 and np.abs(f - want).max() <= 0.5 + 1e-3
        assert (f != s_).mean() < 1e-3
    elif dtype == torch.float32:
        # fp32 end to end.  At these sizes the reference's own fp32 result is 2.4e-5 away from an fp64 evaluation
        # (weights and spans are computed in float), and a different but equally valid rounding of the weights moves
        # single outputs by up to 1.4e-5: the bound is "as close to fp64 as the reference CPU kernel is", plus
        # agreement of our two kernels with each other and with the reference to 3e-5.
        x64 = x.double().cpu().reshape(-1, 1, *x.shape[-2:])
        exact = torch.nn.functional.interpolate(x64, size=list(size), mode="bilinear", antialias=True).numpy().reshape(want.shape)
        err_ref = np.abs(want - exact).max()
        assert np.abs(npy(fast) - exact).max() <= 1.25 * err_ref + 1e-6
        np.testing.assert_allclose(npy(fast), want, rtol=1e-5, atol=3e-5)
        np.testing.assert_allclose(npy(fast), npy(slow), rtol=1e-5, atol=1e-5)
    else:
        np.testing.assert_allclose(npy(fast), want, rtol=1e-2, atol=1e-2)
        np.testing.assert_allclose(npy(fast), npy(slow), rtol=1e-2, atol=4e-3)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16, torch.uint8])
def test_resize_dtypes_shapes_and_identity(vb, oracle, dtype):
    torch.manual_seed(3)
    base = torch.rand(2, 2, 3, 45, 70)
    x = (base * 255).round().to(torch.uint8) if dtype == torch.uint8 else base.to(dtype)
    xd = x.to(DEV)
    for mode, code in (("bilinear", 0), ("bicubic", 1)):
        for aa in (True, False):
            for size in ([20, 31], [90, 100], 30):
                got = vb.transforms.resize_image(xd, size, interpolation=mode, antialias=aa)
                oh, ow = vb.transforms.compute_resized_output_size((45, 70), size)
                assert got.shape == (2, 2, 3, oh, ow) and got.dtype == dtype
                ref = oracle.resize(x.float().numpy(), (oh, ow), code, aa)
                if dtype == torch.uint8:
                    ref = np.rint(np.clip(ref, 0, 255))
                    assert np.abs(npy(got).astype(np.float32) - ref).max() <= 1.0    # rounding ties only
                else:
                    tol = dict(rtol=0, atol=1e-5) if dtype == torch.float32 else dict(rtol=1e-2, atol=1e-2)
                    np.testing.assert_allclose(npy(got), ref, **tol)
    same = vb.transforms.resize_image(xd, [45, 70])
    assert same is xd                                                           # _geometry.py:313-314
    ver = xd._version
    vb.transforms.resize_image(xd, [10, 10])
    assert xd._version == ver                                                   # input never mutated


def _check_roi_align_vs_both_references(ours, ref_cuda, ref_cpu):
    """The reference has TWO implementations that disagree with each other by more than 1e-5 on
    FPN-sized maps: nvcc contracts the sample-coordinate arithmetic of roi_align_kernel.cu:125-135
    into FMAs, the x86 build of cpu/roi_align_kernel.cpp does not, and an ulp of a coordinate ~200 is
    1.5e-5 pixels times the local gradient.  Parity is defined against the CPU kernel (what oracle/
    restates, to 1e-5); against the CUDA kernel we must be no farther than the CPU kernel itself is."""
    np.testing.assert_allclose(ours, ref_cpu, **F32_TOL)
    ref_gap = np.abs(ref_cuda - ref_cpu).max()
    our_gap = np.abs(ours - ref_cuda).max()
    assert our_gap <= ref_gap + 1e-5, (our_gap, ref_gap)


# =============================== drop-in through torchvision ======================
def test_dropin_through_torchvision_api(vb, oracle):
    tv = pytest.importorskip("torchvision")
    from torchvision.transforms.v2 import functional as TF
    from torchvision import tv_tensors
    from vision_b200 import workloads

    x, rois, kw = workloads.cfg2_roi_align(channels=32, k=100)
    xd, rd = x.to(DEV), rois.to(DEV)
    ref_cuda = tv.ops.roi_align(xd, rd, **kw)                                   # reference CUDA kernel (sm_100 SASS)
    vb.install()
    try:
        before = vb.launch_count()
        ours = tv.ops.roi_align(xd, rd, **kw)
        assert vb.launch_count() > before, "torchvision.ops.roi_align did not reach the vision_b200 kernel"
        _check_roi_align_vs_both_references(npy(ours), npy(ref_cuda), npy(tv.ops.roi_align(x, rois, **kw)))
        # autograd still flows through the reference's registered backward
        xg = xd[:, :4].clone().requires_grad_(True)
        tv.ops.roi_align(xg, rd, **kw).sum().backward()
        assert xg.grad is not None and torch.isfinite(xg.grad).all()
        # autocast wrapper casts to fp32 and lands on our CUDA kernel
        with torch.autocast("cuda", dtype=torch.float16):
            y = tv.ops.roi_align(xd.half(), rd.half(), **kw)
        assert y.dtype == torch.float16
        # batched_nms + nms
        b, s, i = workloads.cfg3_batched_nms(n=30_000)
        k1 = tv.ops.batched_nms(b.to(DEV), s.to(DEV), i.to(DEV), 0.5)
        want = oracle.batched_nms(b.numpy(), s.numpy(), i.numpy(), 0.5, mode=oracle.NMS_MODE_CUDA, device_is_cuda=True)
        assert np.array_equal(npy(k1), want)
        k2 = tv.ops.nms(b[:2000].to(DEV), s[:2000].to(DEV), 0.5)
        assert np.array_equal(npy(k2), oracle.nms(b[:2000].numpy(), s[:2000].numpy(), 0.5, oracle.NMS_MODE_CUDA))
        # resize through the v2 functional, incl. tv_tensors
        img = torch.rand(3, 180, 320, device=DEV).half()
        before = vb.launch_count()
        r = TF.resize(tv_tensors.Image(img), [64, 64])
        assert vb.launch_count() > before and isinstance(r, tv_tensors.Image) and r.shape == (3, 64, 64)
        want = torch.from_numpy(oracle.resize(img.float().cpu().numpy(), (64, 64), 0, True)).half().float().numpy()
        np.testing.assert_allclose(npy(r.as_subclass(torch.Tensor)), want, rtol=1e-2, atol=1e-3)
        v = TF.resize(tv_tensors.Video(torch.rand(2, 3, 40, 50, device=DEV)), [20, 20])
        assert v.shape == (2, 3, 20, 20)
    finally:
        vb.uninstall()
    again = tv.ops.roi_align(xd, rd, **kw)
    assert torch.equal(again, ref_cuda)                                          # reference kernel active again


def test_against_reference_cuda_kernels_same_box(vb):
    """Extra: our kernels vs the reference's own CUDA kernels (wheel, sm_100 SASS) on this GPU."""
    tv = pytest.importorskip("torchvision")
    from vision_b200 import workloads

    assert not vb.installed()
    b, s, i = workloads.cfg3_batched_nms(n=100_000)
    bd, sd, idd = b.to(DEV), s.to(DEV), i.to(DEV)
    ref = tv.ops.batched_nms(bd, sd, idd, 0.5)
    ours = vb.ops.batched_nms(bd, sd, idd, 0.5)
    assert torch.equal(ref, ours)                                                # bit-exact vs CUDA reference
    ref = tv.ops.nms(bd[:20000], sd[:20000], 0.5)
    assert torch.equal(ref, vb.ops.nms(bd[:20000], sd[:20000], 0.5))
    x, rois, kw = workloads.cfg2_roi_align(channels=64)
    xd, rd = x.to(DEV), rois.to(DEV)
    _check_roi_align_vs_both_references(npy(vb.ops.roi_align(xd, rd, **kw)), npy(tv.ops.roi_align(xd, rd, **kw)),
                                        npy(tv.ops.roi_align(x, rois, **kw)))
    o1, a1 = torch.ops.torchvision.roi_pool(xd, rd, 0.25, 7, 7)
    o2, a2 = torch.ops.vision_b200.roi_pool(xd, rd, 0.25, 7, 7)
    assert torch.equal(o1, o2) and torch.equal(a1, a2)
    img = torch.rand(4, 3, 540, 960, device=DEV)
    ref = torch.nn.functional.interpolate(img, size=[224, 224], mode="bilinear", antialias=True, align_corners=False)
    np.testing.assert_allclose(npy(vb.transforms.resize(img, [224, 224])), npy(ref), rtol=0, atol=1e-5)


# =============================== the C ABI, directly ================================
def test_c_abi_direct_ctypes_call(vb, oracle):
    """include/vision_b200.h entry point called with raw device pointers — no torch types involved."""
    from vision_b200 import _lib, workloads

    lib = _lib.core()
    x, rois, _ = workloads.cfg2_roi_align(channels=8, k=64)
    xd, rd = x.to(DEV), rois.to(DEV)
    out = torch.empty(64, 8, 7, 7, device=DEV)
    arg = torch.empty(64, 8, 7, 7, device=DEV, dtype=torch.int32)
    stream = torch.cuda.current_stream().cuda_stream
    rc = lib.vb200_roi_pool_forward(ctypes.c_void_p(xd.data_ptr()), ctypes.c_void_p(rd.data_ptr()), ctypes.c_void_p(out.data_ptr()),
                                    ctypes.c_void_p(arg.data_ptr()), 0, 1, 8, 200, 272, 64, 7, 7, ctypes.c_double(0.25),
                                    ctypes.c_void_p(stream))
    assert rc == 0, lib.vb200_last_error()
    torch.cuda.synchronize()
    wo, wa = oracle.roi_pool(x.numpy(), rois.numpy(), 7, 0.25)
    assert np.array_equal(npy(out), wo) and np.array_equal(npy(arg), wa)
    rc = lib.vb200_roi_pool_forward(None, None, None, None, 0, 1, 8, 200, 272, 64, 0, 7, ctypes.c_double(0.25), None)
    assert rc == -1 and b"pooled size" in lib.vb200_last_error()


def test_detection_callers_are_drop_in(vb):
    """The real callers of the path (SURVEY.md §8f): RegionProposalNetwork.filter_proposals (batched_nms over FPN
    levels, rpn.py:242-298), MultiScaleRoIAlign (roi_align per level, poolers.py:147-228) and
    RoIHeads.postprocess_detections (batched_nms over classes, roi_heads.py:680-737), run with the reference kernels
    and again after vision_b200.install(): NMS-driven outputs must be IDENTICAL (bit-exact kept indices), pooled
    features within the roi_align tolerance."""
    tv = pytest.importorskip("torchvision")
    from collections import OrderedDict
    from torchvision.models.detection.anchor_utils import AnchorGenerator
    from torchvision.models.detection.image_list import ImageList
    from torchvision.models.detection.roi_heads import RoIHeads
    from torchvision.models.detection.rpn import RegionProposalNetwork, RPNHead

    torch.manual_seed(0)
    sizes = [(100, 136), (50, 68), (25, 34), (13, 17)]
    feats = OrderedDict((str(i), torch.randn(2, 64, h, w, device=DEV)) for i, (h, w) in enumerate(sizes))
    images = ImageList(torch.zeros(2, 3, 400, 544, device=DEV), [(400, 544), (380, 520)])
    anchors = AnchorGenerator(((32,), (64,), (128,), (256,)), ((0.5, 1.0, 2.0),) * 4)
    rpn = RegionProposalNetwork(anchors, RPNHead(64, 3), 0.7, 0.3, 256, 0.5, dict(training=2000, testing=1000),
                                dict(training=2000, testing=300), 0.7).to(DEV).eval()
    pool = tv.ops.MultiScaleRoIAlign(["0", "1", "2", "3"], 7, 2)
    heads = RoIHeads(pool, None, None, 0.5, 0.5, 512, 0.25, None, 0.01, 0.5, 100)
    logits = torch.randn(600, 21, device=DEV) * 3
    reg = torch.randn(600, 21 * 4, device=DEV) * 0.5

    def run():
        with torch.no_grad():
            props, _ = rpn(images, feats)
            pooled = pool(feats, props, images.image_sizes)
            dets = heads.postprocess_detections(logits, reg, [p[:300] for p in props], images.image_sizes)
        return props, pooled, dets

    assert not vb.installed()
    ref_props, ref_pooled, ref_dets = run()
    vb.install()
    try:
        before = vb.launch_count()
        props, pooled, dets = run()
        assert vb.launch_count() > before            # our kernels ran, not the wheel's
    finally:
        vb.uninstall()
    for a, b in zip(props, ref_props):
        assert a.shape == b.shape and torch.equal(a, b)
    assert pooled.shape == ref_pooled.shape
    # the reference CUDA roi_align is itself up to 7e-5 away from its CPU kernel (see _check_roi_align_vs_both_references)
    cpu_pooled = pool(OrderedDict((k, v.cpu()) for k, v in feats.items()), [p.cpu() for p in ref_props], images.image_sizes)
    torch.testing.assert_close(pooled.cpu(), cpu_pooled, rtol=1e-5, atol=1e-5)
    assert (pooled - ref_pooled).abs().max().item() <= (ref_pooled.cpu() - cpu_pooled).abs().max().item() + 2e-5
    for ours, ref in zip(dets, ref_dets):            # (boxes, scores, labels), each a per-image list
        assert len(ours) == len(ref) == 2
        for a, b in zip(ours, ref):
            assert a.shape == b.shape and torch.equal(a, b)


def test_extra_goldens_from_the_reference(vb, golden_extra):
    """tests/golden/reference_cpu_extra.npz: outputs of the reference itself for the shapes that reach the line-wise
    roi_align kernel, the float64 NMS path and the uint8 / fp32 streaming resize."""
    g = golden_extra
    x, r = t(g["line_x"]), t(g["line_rois"])
    for al in (0, 1):
        for path in ("line", "plane", "generic"):
            with force_env("VB200_ROI_ALIGN_PATH", path):
                got = vb.ops.roi_align(x, r, 7, 0.25, 2, bool(al))
            np.testing.assert_allclose(npy(got), g[f"line_out_a{al}"], **F32_TOL)
    b, s, i = t(g["nms64_boxes"]), t(g["nms64_scores"]), t(g["nms64_idxs"])
    assert b.dtype == torch.float64
    _set(vb, "cpu")                                  # the fixtures come from the CPU kernel's arithmetic
    try:
        for k, thr in enumerate(g["nms64_thr"]):
            assert np.array_equal(npy(vb.ops.nms(b, s, float(thr))), g[f"nms64_keep{k}"])
        assert np.array_equal(npy(vb.ops.batched_nms(b, s, i, 0.5)), g["bnms64_keep_t"])    # numel 2800: coordinate trick
    finally:
        _set(vb, "cuda")
    img = t(g["rs8_img"])
    for size in ((9, 20), (31, 200)):
        want, want_f = g[f"rs8_out_{size[0]}x{size[1]}"], g[f"rs8_float_{size[0]}x{size[1]}"]
        ties = np.abs(want_f - np.floor(want_f) - 0.5) < 1e-3
        for path in ("stream", "generic"):           # anything but "generic" leaves the streaming kernel on
            with force_env("VB200_RESIZE_PATH", path):
                got = npy(vb.transforms.resize_image(img, list(size), antialias=True))
            assert got.dtype == np.uint8 and np.array_equal(got[~ties], want[~ties])
            assert np.abs(got.astype(np.int32) - want.astype(np.int32)).max() <= 1
    got = vb.transforms.resize_image(t(g["rsf_img"]), [20, 60], antialias=True)
    np.testing.assert_allclose(npy(got), g["rsf_out_20x60"], rtol=1e-5, atol=1e-5)
