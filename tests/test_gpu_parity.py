"""GPU parity tests: the CUDA path (through the C ABI in libsln_b200.so) against the CPU oracle
on the same seeded inputs.  Run on the B200 box with `-m gpu`.

Bars (BASELINE.json north_star): NMS keep indices, top-k order, layer planes and EDT squared
distances bit-exact; RoIAlign forward/backward within 1e-5 relative in fp32 -- the kernels here
reproduce the reference's rounding sequence, so the tests additionally require bit-equality
for RoIAlign and report it as such.
"""
import numpy as np
import pytest
import torch

from oracle import oracle
from sln_amodal_b200 import synth

pytestmark = pytest.mark.gpu

RTOL = 1e-5     # north_star tolerance for RoIAlign fwd/bwd (fp32, relative)


def dev():
    return torch.device("cuda", 0)


def cuda(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.to(dev())


def assert_close_rel(got, want, rtol=RTOL):
    got = np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    scale = max(np.abs(want).max(), 1e-30)
    err = np.abs(got - want).max() / scale
    assert err <= rtol, f"max rel err {err:.3e} > {rtol}"


# --------------------------------------------------------------------------- crop forward
def _crop_inputs(seed, B, C, H, W, N, **kw):
    rng = np.random.default_rng(seed)
    img = rng.standard_normal((B, C, H, W), dtype=np.float32)
    boxes = synth.roi_boxes(N, seed=seed + 1, **kw)
    ind = rng.integers(0, B, N).astype(np.int32)
    return img, boxes, ind


@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("C,H,W,N,ph,pw", [
    (256, 64, 64, 300, 7, 7), (256, 32, 32, 200, 14, 14), (256, 64, 64, 100, 16, 16),
    (1, 128, 128, 64, 32, 32), (3, 97, 61, 80, 5, 9), (183, 65, 65, 50, 16, 16),
    (8, 40, 40, 33, 1, 1), (4, 17, 23, 40, 1, 6), (260, 16, 16, 20, 7, 7), (512, 16, 16, 20, 3, 3),
])
def test_crop_forward_matches_oracle(layout, C, H, W, N, ph, pw):
    from sln_amodal_b200 import ops
    img, boxes, ind = _crop_inputs(100 + C + ph, 3, C, H, W, N, outside_frac=0.15, degenerate_frac=0.05)
    for ext in (0.0, -7.25):
        want = oracle.crop_and_resize_fwd(img, boxes, ind, ph, pw, ext)
        t = cuda(img)
        if layout == "nhwc":
            t = t.contiguous(memory_format=torch.channels_last)
        got = ops.crop_and_resize_forward(t, cuda(boxes), cuda(ind), ph, pw, ext)
        assert got.shape == want.shape
        if layout == "nhwc" and C > 1:
            assert got.is_contiguous(memory_format=torch.channels_last)
        g = got.contiguous().cpu().numpy()
        assert_close_rel(g, want)
        assert g.tobytes() == want.tobytes(), "forward is expected to be bit-exact"


def test_crop_forward_special_boxes():
    from sln_amodal_b200 import ops
    img = np.arange(2 * 2 * 5 * 5, dtype=np.float32).reshape(2, 2, 5, 5)
    boxes = np.array([[0, 0, 1, 1], [0.25, 0.25, 0.75, 0.75], [1, 1, 1, 1], [-0.5, 0, 0.5, 1],
                      [0.9, 0.9, 0.1, 0.1], [0, 0, 2, 2], [np.nan, 0, 1, 1]], np.float32)
    ind = np.array([0, 1, 1, 0, 1, 0, 0], np.int32)
    want = oracle.crop_and_resize_fwd(img, boxes[:6], ind[:6], 5, 5, -1.0)
    for cl in (False, True):
        t = cuda(img)
        if cl:
            t = t.contiguous(memory_format=torch.channels_last)
        got = ops.crop_and_resize_forward(t, cuda(boxes), cuda(ind), 5, 5, -1.0).contiguous().cpu().numpy()
        assert got[:6].tobytes() == want.tobytes()
        assert np.all(got[6] == -1.0)        # NaN box: documented as all-extrapolation
    # out-of-range box_ind rows are zeros (reference GPU kernel behaviour), others untouched
    bad = np.array([0, 5, -1, 0, 1, 0, 0], np.int32)
    got = ops.crop_and_resize_forward(cuda(img), cuda(boxes), cuda(bad), 5, 5, -1.0).cpu().numpy()
    assert np.all(got[1] == 0) and np.all(got[2] == 0)
    assert got[0].tobytes() == want[0].tobytes()
    # empty
    e = ops.crop_and_resize_forward(cuda(img), cuda(np.zeros((0, 4), np.float32)), cuda(np.zeros(0, np.int32)), 7, 7)
    assert tuple(e.shape) == (0, 2, 7, 7)


# --------------------------------------------------------------------------- crop backward
@pytest.mark.parametrize("C,H,W,N,ph,pw,kw", [
    (256, 32, 32, 150, 7, 7, {}), (256, 64, 64, 120, 14, 14, {}), (64, 48, 40, 90, 16, 16, {}),
    (3, 31, 29, 60, 5, 4, {}), (130, 20, 20, 40, 7, 7, {}), (8, 33, 33, 50, 1, 1, {}),
    (32, 64, 64, 400, 7, 7, {"window": (0.5, 0.5, 0.06)}),      # all ROIs inside one small window
    (16, 24, 24, 0, 7, 7, {}),                                   # no ROIs: pure zero fill
])
def test_crop_backward_bit_exact(C, H, W, N, ph, pw, kw):
    from sln_amodal_b200 import ops
    B = 3
    rng = np.random.default_rng(7 + C + N)
    boxes = synth.roi_boxes(N, seed=11 + N, outside_frac=0.1, degenerate_frac=0.05, **kw) if N else np.zeros((0, 4), np.float32)
    ind = rng.integers(0, B, N).astype(np.int32)
    g = rng.standard_normal((N, C, ph, pw), dtype=np.float32)
    want = oracle.crop_and_resize_bwd(g, boxes, ind, (B, C, H, W))
    for cl in (True, False):
        gt = cuda(g)
        if cl:
            gt = gt.contiguous(memory_format=torch.channels_last)
        # exact mode: the reference's rounding sequence and summation order -> bit-identical
        got = ops.crop_and_resize_backward(gt, cuda(boxes), cuda(ind), (B, C, H, W), exact=True)
        gn = got.contiguous().cpu().numpy()
        assert gn.tobytes() == want.tobytes(), "exact backward must be bit-identical to crop_and_resize.c"
        # default mode: fma per term, same order -> within the 1e-5 bar (in practice ~1e-7)
        got = ops.crop_and_resize_backward(gt, cuda(boxes), cuda(ind), (B, C, H, W), exact=False)
        gn = got.contiguous().cpu().numpy()
        assert_close_rel(gn, want)
        assert_close_rel(gn, want, rtol=2e-6)
        assert np.array_equal(gn == 0, want == 0) or np.abs(gn[(gn == 0) != (want == 0)]).max() < 1e-30


def test_crop_backward_deterministic():
    from sln_amodal_b200 import ops
    rng = np.random.default_rng(3)
    N, C, H, W, B = 600, 256, 32, 32, 2
    boxes = cuda(synth.roi_boxes(N, seed=5, window=(0.5, 0.5, 0.5)))
    ind = cuda(rng.integers(0, B, N).astype(np.int32))
    g = cuda(rng.standard_normal((N, C, 7, 7), dtype=np.float32)).contiguous(memory_format=torch.channels_last)
    for exact in (False, True):
        a = ops.crop_and_resize_backward(g, boxes, ind, (B, C, H, W), exact=exact)
        for _ in range(3):
            b = ops.crop_and_resize_backward(g, boxes, ind, (B, C, H, W), exact=exact)
            assert torch.equal(a, b)


def test_nchw_maps_take_the_nhwc_kernel_through_a_remembered_copy():
    """NCHW images with >= 32 channels (what the unmodified reference passes) are transposed once and the copy is
    remembered while the tensor lives: the result must track in-place updates, views of the same storage, and a new
    tensor that reuses the address of a dead one."""
    import gc
    from sln_amodal_b200 import ops
    img, boxes, ind = _crop_inputs(77, 2, 64, 40, 48, 120, outside_frac=0.1)
    tb, ti = cuda(boxes), cuda(ind)
    t = cuda(img)
    assert t.is_contiguous()
    for _ in range(2):                                              # second call: served from the remembered copy
        got = ops.crop_and_resize_forward(t, tb, ti, 7, 7)
        assert got.is_contiguous(memory_format=torch.channels_last)
        assert got.contiguous().cpu().numpy().tobytes() == oracle.crop_and_resize_fwd(img, boxes, ind, 7, 7).tobytes()
    t.mul_(2.0)                                                     # in-place update bumps the version counter
    got = ops.crop_and_resize_forward(t, tb, ti, 7, 7)
    assert got.contiguous().cpu().numpy().tobytes() == oracle.crop_and_resize_fwd(img * 2, boxes, ind, 7, 7).tobytes()
    v = t[1:2]                                                      # a view of the same storage (other offset / shape)
    got = ops.crop_and_resize_forward(v, tb, torch.zeros_like(ti), 5, 5)
    want = oracle.crop_and_resize_fwd(img[1:2] * 2, boxes, np.zeros_like(ind), 5, 5)
    assert got.contiguous().cpu().numpy().tobytes() == want.tobytes()
    sq = t[0].unsqueeze(0)                                          # the reference's squeeze(0) / unsqueeze(0) dance
    got = ops.crop_and_resize_forward(sq, tb, torch.zeros_like(ti), 5, 5)
    assert got.contiguous().cpu().numpy().tobytes() == oracle.crop_and_resize_fwd(img[0:1] * 2, boxes, np.zeros_like(ind), 5, 5).tobytes()
    ptr0 = t.data_ptr()
    del t, v, sq, got
    gc.collect()
    img2 = np.random.default_rng(5).standard_normal(img.shape, dtype=np.float32)
    t2 = cuda(img2)                                                 # usually lands on the freed block
    got = ops.crop_and_resize_forward(t2, tb, ti, 7, 7)
    assert got.contiguous().cpu().numpy().tobytes() == oracle.crop_and_resize_fwd(img2, boxes, ind, 7, 7).tobytes(), (ptr0 == t2.data_ptr())


def test_autograd_function_api():
    from roialign.roi_align.crop_and_resize import CropAndResizeFunction, CropAndResize
    img, boxes, ind = _crop_inputs(9, 2, 16, 24, 24, 30)
    for cl in (False, True):
        t = cuda(img)
        if cl:
            t = t.contiguous(memory_format=torch.channels_last)
        t.requires_grad_(True)
        out = CropAndResizeFunction(7, 7, 0)(t, cuda(boxes), cuda(ind))
        w = cuda(np.random.default_rng(1).standard_normal(out.shape, dtype=np.float32))
        (out * w).sum().backward()
        want_f = oracle.crop_and_resize_fwd(img, boxes, ind, 7, 7, 0.0)
        want_b = oracle.crop_and_resize_bwd(w.cpu().numpy(), boxes, ind, img.shape)
        assert out.detach().contiguous().cpu().numpy().tobytes() == want_f.tobytes()
        assert t.grad.shape == t.shape
        assert_close_rel(t.grad.contiguous().cpu().numpy(), want_b)
        out2 = CropAndResize(7, 7, 0)(t.detach(), cuda(boxes), cuda(ind))
        assert torch.equal(out2, out.detach())


def test_layout_converters_roundtrip():
    from sln_amodal_b200 import ops
    x = torch.randn(3, 37, 19, 23, device=dev())
    cl = ops.to_channels_last(x)
    assert cl.is_contiguous(memory_format=torch.channels_last) and torch.equal(cl, x)
    back = ops.to_contiguous_nchw(cl)
    assert back.is_contiguous() and torch.equal(back, x)


# --------------------------------------------------------------------------- pyramid
def test_pyramid_roi_align_matches_oracle():
    from sln_amodal_b200 import pyramid_roi_align
    rng = np.random.default_rng(21)
    C = 64
    maps = [rng.standard_normal((1, C, s, s), dtype=np.float32) for s in (64, 32, 16, 8)]
    boxes = synth.roi_boxes(300, seed=77)
    levels = oracle.roi_levels(boxes, (256, 256))
    # keep ROIs away from exact level boundaries (log on GPU vs CPU may differ by an ulp there)
    b = boxes.astype(np.float64)
    raw = 4 + np.log2(np.sqrt((b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1])) / (224.0 / 256.0))
    ok = np.abs(raw - np.floor(raw) - 0.5) > 1e-3
    boxes, levels = boxes[ok], levels[ok]
    for pool in (7, 14):
        want = oracle.pyramid_roi_align(boxes, maps, pool, (256, 256), levels=levels)
        tm = [cuda(m).requires_grad_(True) for m in maps]
        got = pyramid_roi_align([cuda(boxes).unsqueeze(0)] + tm, pool, (256, 256, 3))
        assert got.detach().contiguous().cpu().numpy().tobytes() == want.tobytes()
        w = rng.standard_normal(want.shape, dtype=np.float32)
        (got * cuda(w)).sum().backward()
        for i, lvl in enumerate(range(2, 6)):
            ix = np.nonzero(levels == lvl)[0]
            wb = oracle.crop_and_resize_bwd(w[ix], boxes[ix], np.zeros(ix.size, np.int32), maps[i].shape)
            assert_close_rel(tm[i].grad.contiguous().cpu().numpy(), wb, rtol=2e-6)


def test_roi_level_kernel_matches_the_torch_expression():
    """sln_roi_levels against the reference's torch expression (modals.py:53-64) evaluated on the same CUDA tensor
    and against the oracle (torch CPU), incl. zero-area, inverted and non-finite boxes."""
    from sln_amodal_b200 import ops
    from sln_amodal_b200.pyramid import log2
    rng = np.random.default_rng(77)
    boxes = synth.roi_boxes(20000, seed=78)
    boxes[:50, 2] = boxes[:50, 0]                      # zero height
    boxes[50:100, [0, 2]] = boxes[50:100, [2, 0]]      # inverted
    boxes[100, 0] = np.nan
    boxes[101, 3] = np.inf
    # boxes sitting on level boundaries: sqrt(h*w) = 224 * 2^(k-4) / 1024
    for j, k in enumerate((2.5, 3.5, 4.5)):
        side = np.float32(224.0 * 2.0 ** (k - 4) / 1024.0)
        boxes[200 + j] = (0.1, 0.1, np.float32(0.1) + side, np.float32(0.1) + side)
    for hw in ((1024, 1024), (768, 1280)):
        t = cuda(boxes)
        y1, x1, y2, x2 = t.chunk(4, dim=1)
        area = torch.tensor([float(hw[0] * hw[1])], dtype=torch.float32, device=dev())
        want = (4 + log2(torch.sqrt((y2 - y1) * (x2 - x1)) / (224.0 / torch.sqrt(area)))).round().int().clamp(2, 5).view(-1) - 2
        got = ops.roi_levels_device(t, hw)
        assert torch.equal(got, want)
        fin = np.isfinite(boxes).all(1)
        assert np.array_equal(got.cpu().numpy()[fin] + 2, oracle.roi_levels(boxes[fin], hw))


# --------------------------------------------------------------------------- NMS
@pytest.mark.parametrize("kind", ["rpn", "uniform"])
@pytest.mark.parametrize("n", [1, 2, 63, 64, 65, 129, 1000, 2500, 6000])
@pytest.mark.parametrize("ties", [False, True])
def test_nms_bit_exact(kind, n, ties):
    from nms.nms_wrapper import nms
    boxes = synth.nms_boxes(n, seed=7 + n, kind=kind)
    scores = synth.nms_scores(n, seed=8 + n, ties=ties)
    dets = np.concatenate([boxes, scores[:, None]], 1)
    for thr in (0.7, 0.3):
        want = oracle.nms(dets, thr)
        got = nms(cuda(dets), thr)
        assert got.dtype == torch.int64 and got.is_cuda
        assert np.array_equal(got.cpu().numpy(), want)


def test_nms_12k_and_max_keep():
    from sln_amodal_b200 import ops
    n = 12000
    dets = np.concatenate([synth.nms_boxes(n, seed=9), synth.nms_scores(n, seed=10)[:, None]], 1)
    want = oracle.nms(dets, 0.7)
    keep, num = ops.nms_device(cuda(dets), 0.7)
    k = int(num.item())
    assert np.array_equal(keep[:k].cpu().numpy(), want)
    keep, num = ops.nms_device(cuda(dets), 0.7, max_keep=1000)
    k = int(num.item())
    assert k == min(1000, want.size) and np.array_equal(keep[:k].cpu().numpy(), want[:k])


def test_nms_near_threshold_pairs():
    """Pairs engineered to sit within a few ulp of the threshold: the fast sign test must hand
    them to the exact divide and agree with nms.c."""
    from nms.nms_wrapper import nms
    rng = np.random.default_rng(4)
    n = 4000
    base = np.array([100.0, 100.0, 299.0, 299.0], np.float32)       # 200x200 (+1 convention)
    boxes = np.tile(base, (n, 1))
    # shift along x so that inter/union is ~0.7: inter = (200-s)*200, union = (200+s)*200 -> s ~ 35.29
    s = (35.294117 + rng.uniform(-2e-4, 2e-4, n)).astype(np.float32)
    boxes[1:, 1] += s[1:]
    boxes[1:, 3] += s[1:]
    boxes[1:, 0] += (rng.integers(0, 2, n - 1) * 1000).astype(np.float32)   # half of them far away in y
    boxes[1:, 2] = boxes[1:, 0] + 199.0
    scores = synth.nms_scores(n, seed=12)
    scores[0] = 2.0
    dets = np.concatenate([boxes, scores[:, None]], 1).astype(np.float32)
    want = oracle.nms(dets, 0.7)
    got = nms(cuda(dets), 0.7).cpu().numpy()
    assert np.array_equal(got, want)


def test_nms_long_dependency_chain_takes_serial_fallback():
    """A chain where box k only overlaps box k+1 needs ~n rounds of the parallel fixed-point resolve;
    it must fall back to the serial scan and still be exact."""
    from nms.nms_wrapper import nms
    n = 10400                               # >= 160 words: takes the parallel resolve first
    w, s = 100.0, 12.0                      # IoU(k,k+1) = 88/112 = 0.786 >= 0.7, IoU(k,k+2) = 76/124 < 0.7
    k = np.arange(n, dtype=np.float32)
    boxes = np.stack([np.zeros(n, np.float32), k * s, np.full(n, 49.0, np.float32), k * s + w - 1], 1)
    scores = np.linspace(1.0, 0.0, n).astype(np.float32)
    dets = np.concatenate([boxes, scores[:, None]], 1).astype(np.float32)
    want = oracle.nms(dets, 0.7)
    assert np.array_equal(want, np.arange(0, n, 2))
    assert np.array_equal(nms(cuda(dets), 0.7).cpu().numpy(), want)


def test_nms_two_stage_path_20k():
    from sln_amodal_b200 import ops
    n = 20000
    dets = np.concatenate([synth.nms_boxes(n, seed=21), synth.nms_scores(n, seed=22)[:, None]], 1)
    want = oracle.nms(dets, 0.7)
    keep, num = ops.nms_device(cuda(dets), 0.7)
    assert np.array_equal(keep[: int(num.item())].cpu().numpy(), want)
    keep, num = ops.nms_device(cuda(dets), 0.7, max_keep=500)
    assert np.array_equal(keep[: int(num.item())].cpu().numpy(), want[:500])


def test_nms_empty_and_degenerate():
    from nms.nms_wrapper import nms
    assert nms(torch.zeros((0, 5), device=dev()), 0.5).numel() == 0
    dets = np.array([[10, 10, 5, 5, 0.9], [10, 10, 5, 5, 0.8], [0, 0, 0, 0, 0.7], [0, 0, 0, 0, 0.7],
                     [3, 3, 8, 8, np.float32(0.5)]], np.float32)      # inverted and zero-size boxes, tied scores
    for thr in (0.0, 0.3, 1.0):
        assert np.array_equal(nms(cuda(dets), thr).cpu().numpy(), oracle.nms(dets, thr))


def _nms_both_paths(dets, thr, cls=None, max_keep=0):
    """(sparse-or-whatever-ran result, dense-only result, path flag) as numpy."""
    from sln_amodal_b200 import ops
    d = cuda(dets)
    c = None if cls is None else cuda(cls)
    keep, num, path = ops.nms_device(d, thr, class_ids=c, max_keep=max_keep, return_path=True)
    keep_d, num_d = ops.nms_device(d, thr, class_ids=c, max_keep=max_keep, dense_only=True)
    return (keep[: int(num.item())].cpu().numpy(), keep_d[: int(num_d.item())].cpu().numpy(), int(path.item()))


@pytest.mark.parametrize("kind,n,thr,sparse", [
    ("rpn", 65, 0.7, True), ("rpn", 1000, 0.7, True), ("rpn", 12000, 0.7, True), ("uniform", 12000, 0.7, True),
    ("rpn", 6000, 0.5, None), ("rpn", 6000, 0.3, None), ("uniform", 6000, 0.3, True), ("rpn", 4000, 0.05, None),
    ("uniform", 4000, 0.05, None), ("rpn", 3000, 0.95, True), ("rpn", 3000, 1.0, True), ("rpn", 40000, 0.7, None), ("uniform", 40000, 0.7, True),
    ("uniform", 65535, 0.6, True)])
def test_nms_sparse_path_equals_dense_and_oracle(kind, n, thr, sparse):
    """The binned pipeline must take the inputs marked True (path == 1) -- the others may exceed its edge budget and
    hand over to the dense kernels on the device -- and always agree with the dense bit-matrix pipeline; up to 12k
    boxes both are also checked against nms.c."""
    dets = np.concatenate([synth.nms_boxes(n, seed=31 + n, kind=kind), synth.nms_scores(n, seed=32 + n)[:, None]], 1)
    got, dense, path = _nms_both_paths(dets, thr)
    assert path == 1 or not sparse
    assert np.array_equal(got, dense)
    if n <= 12000:
        assert np.array_equal(got, oracle.nms(dets, thr))
    got, dense, path = _nms_both_paths(dets, thr, max_keep=100)
    assert (path == 1 or not sparse) and np.array_equal(got, dense) and got.size <= 100


def test_nms_sparse_path_offsets_and_scales():
    """Windows are relative to the box size and the grid to the centres' bounding box: translated, huge and tiny
    boxes (still inside +-32768) must stay on the sparse path and agree with nms.c."""
    n = 3000
    base = synth.nms_boxes(n, seed=5)
    sc = synth.nms_scores(n, seed=6)
    for scale, shift in ((1.0, -20000.0), (30.0, 0.0), (1.0 / 8, 0.0), (1.0 / 512, 0.0), (1.0, 31000.0)):
        dets = np.concatenate([(base * scale + shift).astype(np.float32), sc[:, None]], 1)
        got, dense, path = _nms_both_paths(dets, 0.7)
        assert path == 1 or scale < 1.0          # sub-pixel boxes all overlap under the +1 convention: may bail out
        assert np.array_equal(got, dense) and np.array_equal(got, oracle.nms(dets, 0.7))


def test_nms_sparse_path_bails_out_to_dense():
    """Outside the sparse contract the dense kernels must produce the result: heavy duplication (more than
    16 n overlapping pairs), non-finite / inverted / far-away boxes, tiny thresholds."""
    rng = np.random.default_rng(11)
    n = 2000
    sc = synth.nms_scores(n, seed=13)
    # (a) 2000 near-identical boxes: ~n^2/2 edges
    boxes = (np.array([100, 100, 300, 300], np.float32) + rng.normal(0, 1.0, (n, 4))).astype(np.float32)
    dets = np.concatenate([boxes, sc[:, None]], 1)
    got, dense, path = _nms_both_paths(dets, 0.7)
    assert path == 0 and np.array_equal(got, dense) and np.array_equal(got, oracle.nms(dets, 0.7))
    # (b) one inverted box / one NaN / one inf / one far outside the coordinate bound
    base = synth.nms_boxes(n, seed=14)
    for bad in ([50, 50, 10, 10], [np.nan, 0, 10, 10], [0, 0, np.inf, 10], [0, 0, 10, 40000.0]):
        b = base.copy()
        b[777] = np.array(bad, np.float32)
        dets = np.concatenate([b, sc[:, None]], 1)
        got, dense, path = _nms_both_paths(dets, 0.7)
        assert path == 0 and np.array_equal(got, dense)
        if np.isfinite(b).all():
            assert np.array_equal(got, oracle.nms(dets, 0.7))
    # (c) thresholds below 0.05 (and NaN) are dense by construction
    dets = np.concatenate([base, sc[:, None]], 1)
    for thr in (0.0, 0.01, -1.0):
        got, dense, path = _nms_both_paths(dets, thr)
        assert path == 0 and np.array_equal(got, oracle.nms(dets, thr))


def test_nms_sparse_vs_dense_random_configs():
    """Randomised sweep over sizes, thresholds, box statistics, score ties and class counts: whatever pipeline runs must
    agree with the dense bit-matrix pipeline (and with nms.c on the smaller cases)."""
    rng = np.random.default_rng(2025)
    for case in range(24):
        n = int(rng.choice([65, 66, 100, 257, 511, 1024, 3000, 7777]))
        thr = float(rng.choice([0.05, 0.1, 0.3, 0.5, 0.7, 0.9]))
        kind = "rpn" if rng.random() < 0.6 else "uniform"
        boxes = synth.nms_boxes(n, seed=1000 + case, kind=kind, rounded=bool(rng.random() < 0.3))
        if rng.random() < 0.25:                                   # collapse the centres onto a line / a point
            boxes[:, [1, 3]] = boxes[:1, [1, 3]]
        scores = synth.nms_scores(n, seed=2000 + case, ties=bool(rng.random() < 0.5))
        dets = np.concatenate([boxes, scores[:, None]], 1).astype(np.float32)
        cls = None
        if rng.random() < 0.4:
            cls = rng.integers(-3, int(rng.choice([2, 7, 200])), n).astype(np.int32)
        got, dense, path = _nms_both_paths(dets, thr, cls=cls)
        assert np.array_equal(got, dense), (case, n, thr, kind, path)
        if cls is None and n <= 3000:
            assert np.array_equal(got, oracle.nms(dets, thr)), (case, n, thr, kind, path)


def test_nms_sparse_only_flag_and_host_retry():
    """SLN_NMS_SPARSE_ONLY: the sparse pipeline alone; num_keep = -1 reports a bail-out, and the reference-facing
    nms() retries with the dense pipeline."""
    from sln_amodal_b200 import ops
    from nms.nms_wrapper import nms
    n = 5000
    sc = synth.nms_scores(n, seed=51)
    dets = np.concatenate([synth.nms_boxes(n, seed=50), sc[:, None]], 1)
    want = oracle.nms(dets, 0.7)
    keep, num = ops.nms_device(cuda(dets), 0.7, sparse_only=True)
    assert int(num.item()) == want.size and np.array_equal(keep[: want.size].cpu().numpy(), want)
    keep, num = ops.nms_device(cuda(dets), 0.7, sparse_only=True, max_keep=37)
    assert int(num.item()) == 37 and np.array_equal(keep[:37].cpu().numpy(), want[:37])
    # heavy duplication: outside the sparse contract
    rng = np.random.default_rng(52)
    dup = np.concatenate([(np.array([100, 100, 300, 300], np.float32) + rng.normal(0, 1.0, (n, 4))).astype(np.float32), sc[:, None]], 1)
    keep, num = ops.nms_device(cuda(dup), 0.7, sparse_only=True)
    assert int(num.item()) == -1
    assert np.array_equal(nms(cuda(dup), 0.7).cpu().numpy(), oracle.nms(dup, 0.7))
    # inputs the sparse pipeline never attempts run dense even with the flag
    keep, num = ops.nms_device(cuda(dets), 0.01, sparse_only=True)
    w2 = oracle.nms(dets, 0.01)
    assert int(num.item()) == w2.size and np.array_equal(keep[: w2.size].cpu().numpy(), w2)


def test_nms_sparse_resolve_is_interleaving_independent():
    """The resolve kernel lets warps read the known-kept / known-dead sets while other CTAs extend them (the hazards
    compute-sanitizer's racecheck reports; soundness argument in nms.cu above nms_sparse_resolve_kernel).  The hardware
    interleaving differs from launch to launch: 320 launches over four inputs the sparse pipeline takes (clustered RPN-like
    boxes with multi-round suppression chains, a low-overlap set, a high threshold) must all return the oracle's survivors."""
    from sln_amodal_b200 import ops
    cases = []
    for n, seed, kind, thr in ((12000, 71, "rpn", 0.7), (4000, 72, "rpn", 0.7), (12000, 73, "uniform", 0.7), (3000, 74, "rpn", 0.95)):
        cases.append((np.concatenate([synth.nms_boxes(n, seed=seed, kind=kind), synth.nms_scores(n, seed=seed + 1)[:, None]], 1), thr))
    streams = [torch.cuda.Stream() for _ in range(2)]
    for dets, thr in cases:
        want = oracle.nms(dets, thr)
        d = cuda(dets)
        ref_keep, ref_num = ops.nms_device(d, thr, sparse_only=True)
        assert int(ref_num.item()) == want.size and np.array_equal(ref_keep[: want.size].cpu().numpy(), want)
        torch.cuda.synchronize()
        for it in range(80):
            # a second stream keeps other kernels in flight so that CTA placement and timing vary between launches
            with torch.cuda.stream(streams[it % 2]):
                noise = torch.randn(1 << (12 + it % 8), device=d.device).sum()
            keep, num = ops.nms_device(d, thr, sparse_only=True)
            assert int(num.item()) == want.size, (it, int(num.item()))
            assert torch.equal(keep[: want.size], ref_keep[: want.size]), it
            del noise
        torch.cuda.synchronize()


def test_nms_sparse_chain_falls_back():
    """A 3000-long dependency chain exceeds the sparse resolve's round budget: dense takes over, still exact."""
    n = 3000
    k = np.arange(n, dtype=np.float32)
    boxes = np.stack([np.zeros(n, np.float32), k * 12.0, np.full(n, 49.0, np.float32), k * 12.0 + 99.0], 1)
    dets = np.concatenate([boxes, np.linspace(1.0, 0.0, n, dtype=np.float32)[:, None]], 1).astype(np.float32)
    got, dense, path = _nms_both_paths(dets, 0.7)
    assert path == 0 and np.array_equal(got, np.arange(0, n, 2)) and np.array_equal(dense, got)


@pytest.mark.parametrize("K,n,thr", [(81, 12000, 0.3), (61, 12000, 0.3), (5, 5000, 0.5), (1000, 8000, 0.3)])
def test_nms_sparse_class_aware_equals_dense(K, n, thr):
    rng = np.random.default_rng(K + n)
    boxes = synth.nms_boxes(n, seed=40 + K, rounded=True)
    dets = np.concatenate([boxes, synth.nms_scores(n, seed=41 + K)[:, None]], 1)
    cls = (rng.integers(0, K, n) - K // 2).astype(np.int32)          # negative ids too
    got, dense, path = _nms_both_paths(dets, thr, cls=cls)
    assert path == 1 and np.array_equal(got, dense)
    want = oracle.per_class_nms(boxes, cls, dets[:, 4].copy(), thr)
    assert np.array_equal(np.sort(got), want)


@pytest.mark.parametrize("K,n", [(81, 3000), (61, 12000)])
def test_per_class_nms_matches_reference_loop(K, n):
    from sln_amodal_b200 import batched_nms
    rng = np.random.default_rng(K)
    boxes = synth.nms_boxes(n, seed=9 + K, rounded=True)
    scores = synth.nms_scores(n, seed=8 + K)
    cls = rng.integers(1, K, n).astype(np.int32)
    want = oracle.per_class_nms(boxes, cls, scores, 0.3)
    got = batched_nms(cuda(boxes), cuda(scores), cuda(cls), 0.3).cpu().numpy()
    assert np.array_equal(np.sort(got), want)
    assert np.all(np.diff(scores[got]) <= 0)


def test_nms_and_proposal_replay_from_a_cuda_graph():
    """Every entry point is stream-ordered with no host round trip, so a call can be captured once in a CUDA graph
    and replayed on new data in the same buffers (cluster launches, the cooperative launch and the memsets included)."""
    from sln_amodal_b200 import ops
    n = 3000
    dets = cuda(np.concatenate([synth.nms_boxes(n, seed=60), synth.nms_scores(n, seed=61)[:, None]], 1))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.nms_device(dets, 0.7)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        keep, num = ops.nms_device(dets, 0.7)
    for seed in (62, 63):                     # new boxes and scores in the captured input buffer
        new = np.concatenate([synth.nms_boxes(n, seed=seed, kind="uniform" if seed == 63 else "rpn"),
                              synth.nms_scores(n, seed=seed + 10)[:, None]], 1).astype(np.float32)
        dets.copy_(torch.from_numpy(new))
        g.replay()
        torch.cuda.synchronize()
        want = oracle.nms(new, 0.7)
        assert int(num.item()) == want.size and np.array_equal(keep[: want.size].cpu().numpy(), want)


@pytest.mark.parametrize("min_conf", [0.0, 0.3])
@pytest.mark.parametrize("n,K", [(1000, 81), (300, 61), (40, 2)])
def test_refine_detections_fused_matches_oracle(n, K, min_conf):
    """The fused front (sln_refine_decode) + class-aware NMS against the oracle's restatement of
    refine_detections (Functions.py:453-557): same detections, same order, same keep indices."""
    from sln_amodal_b200 import refine_detections
    rng = np.random.default_rng(n + K)
    rois = synth.roi_boxes(n, seed=n)
    logits = rng.standard_normal((n, K)).astype(np.float32) * 3.0
    probs = (np.exp(logits) / np.exp(logits).sum(1, keepdims=True)).astype(np.float32)
    probs[:5] = probs[0]                                   # exact ties across rows
    probs[5, :] = np.float32(1.0 / K)                      # tie inside a row: first maximum wins (class 0 -> filtered)
    deltas = (rng.standard_normal((n, K, 4)) * 0.3).astype(np.float32)
    window = (0.0, 0.0, 1024.0, 1024.0)

    class Cfg:
        RPN_BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
        IMAGE_SHAPE = np.array([1024, 1024, 3])
        USE_NMS = True
        DETECTION_MIN_CONFIDENCE = min_conf
        DETECTION_NMS_THRESHOLD = 0.3

    want_det, want_keep = oracle.refine_detections(rois, probs, deltas, window, min_confidence=min_conf, nms_threshold=0.3)
    det, keep = refine_detections(cuda(rois), cuda(probs), cuda(deltas), window, Cfg())
    if want_keep.size == 0:
        assert len(det) == 0
        return
    assert np.array_equal(keep.cpu().numpy(), want_keep)
    assert np.array_equal(det.cpu().numpy(), want_det)


@pytest.mark.parametrize("n,K,bg_frac", [(1000, 81, 0.0), (1000, 2, 0.5), (5000, 61, 0.0), (257, 3, 0.3), (60, 2, 0.0), (40, 4, 1.0)])
def test_refine_detections_without_nms_matches_oracle(n, K, bg_frac):
    """USE_NMS = False -- the reference's shipped default (config.py:78; Functions.py:526-546): decode + device top-100
    (sln_refine_decode + sln_refine_topk) against the oracle: same rows, same order, same keep indices; score ties
    (rows 0-4 and a block of quantised scores) go to the lower ROI index; DETECTION_MIN_CONFIDENCE is ignored here."""
    from sln_amodal_b200 import refine_detections
    rng = np.random.default_rng(7 * n + K)
    rois = synth.roi_boxes(n, seed=n + 1)
    logits = rng.standard_normal((n, K)).astype(np.float32) * 3.0
    bg = rng.random(n) < bg_frac
    logits[bg, 0] = 50.0                                   # background wins: filtered
    probs = (np.exp(logits - logits.max(1, keepdims=True)) / np.exp(logits - logits.max(1, keepdims=True)).sum(1, keepdims=True)).astype(np.float32)
    probs[:5] = probs[0]                                   # exact ties across rows
    q = slice(n // 2, n // 2 + 40)
    probs[q] = np.round(probs[q] * 8) / 8                  # many equal winning scores around the cut
    deltas = (rng.standard_normal((n, K, 4)) * 0.3).astype(np.float32)
    window = (0.0, 0.0, 1024.0, 1024.0)

    class Cfg:
        RPN_BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
        IMAGE_SHAPE = np.array([1024, 1024, 3])
        USE_NMS = False
        DETECTION_MIN_CONFIDENCE = 0.7                     # must NOT filter on this branch (:492-495)
        DETECTION_NMS_THRESHOLD = 0.3

    want_det, want_keep = oracle.refine_detections(rois, probs, deltas, window, use_nms=False)
    det, keep = refine_detections(cuda(rois), cuda(probs), cuda(deltas), window, Cfg())
    if want_keep.size == 0:
        assert len(det) == 0 and len(keep) == 0
        return
    assert want_keep.size <= 100
    assert np.array_equal(keep.cpu().numpy(), want_keep)
    assert det.cpu().numpy().tobytes() == want_det.tobytes()


def test_nms_at_exactly_the_threshold_follows_the_cpu_extension():
    """The reference's two NMS builds disagree at IoU == thresh: cpu_nms suppresses (`ovr >= thresh`, nms.c:58-61), the CUDA
    kernel keeps (`> thresh`, nms_kernel.cu:63).  This library implements the CPU extension's rule -- the oracle the north
    star names -- on CUDA tensors too.  Rounded pixel boxes (refine_detections, Functions.py:485) hit the case exactly:
    10x10 boxes (the +1 convention) shifted by 5 columns overlap with IoU 50 / 150 = 1/3, exactly representable ratios
    are rarer, so thresholds are taken from the computed float."""
    from sln_amodal_b200 import nms
    a = np.array([[0, 0, 9, 9, 0.9], [0, 5, 9, 14, 0.8], [50, 50, 59, 59, 0.7]], np.float32)
    iou = np.float32(np.float32(50.0) / np.float32(100.0 + 100.0 - 50.0))
    keep_at = nms(cuda(a), float(iou)).cpu().numpy()
    assert np.array_equal(keep_at, oracle.nms(a, float(iou))) and np.array_equal(keep_at, [0, 2])      # suppressed at equality
    above = float(np.nextafter(iou, np.float32(1.0)))
    keep_above = nms(cuda(a), above).cpu().numpy()
    assert np.array_equal(keep_above, oracle.nms(a, above)) and np.array_equal(keep_above, [0, 1, 2])


def test_unmold_detections_drops_boxes_the_reference_cannot_paste():
    """A detection whose box leaves the image after the window transform (or is turned inside out) makes the reference's
    paste raise; here it is dropped with its class and score, so the four outputs stay consistent."""
    from sln_amodal_b200 import unmold
    rng = np.random.default_rng(2)
    det = np.array([[10, 10, 60, 70, 1, 0.9], [90, 20, 130, 60, 1, 0.8], [70, 60, 40, 20, 1, 0.7], [5, 5, 50, 50, 1, 0.6]], np.float32)
    masks = rng.random((4, 28, 28, 2)).astype(np.float32)
    boxes, class_ids, scores, planes = unmold.unmold_detections(det, masks, (128, 128, 3), (0, 0, 128, 128))
    assert boxes.tolist() == [[10, 10, 60, 70], [5, 5, 50, 50]] and scores.tolist() == [np.float32(0.9), np.float32(0.6)]
    assert planes.shape == (128, 128, 2)
    for k, i in enumerate((0, 3)):
        assert np.array_equal(planes[:, :, k], oracle.unmold_mask(masks[i, :, :, 1], det[i, :4].astype(np.int32), (128, 128, 3)))


# --------------------------------------------------------------------------- proposal layer
class _Cfg:
    RPN_BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
    IMAGE_SHAPE = np.array([1024, 1024, 3])
    GPU_COUNT = 1


def _proposal_inputs(A, seed, ties=False):
    rng = np.random.default_rng(seed)
    cy, cx = rng.uniform(0, 1024, A), rng.uniform(0, 1024, A)
    h = np.exp(rng.uniform(np.log(16), np.log(512), A))
    w = h * np.exp(rng.uniform(np.log(0.5), np.log(2), A))
    anchors = np.stack([cy - h / 2, cx - w / 2, cy + h / 2, cx + w / 2], 1).astype(np.float32)
    fg = rng.permutation(np.linspace(0.0, 1.0, A)).astype(np.float32)
    if ties:
        fg = (np.floor(fg * 500) / 500).astype(np.float32)
    probs = np.stack([1 - fg, fg], 1).astype(np.float32)
    deltas = (rng.standard_normal((A, 4)) * np.array([1.0, 1.0, 1.5, 1.5])).astype(np.float32)
    return probs, deltas, anchors


@pytest.mark.parametrize("A,count,ties", [(261888, 1000, False), (261888, 2000, True), (20000, 1000, True),
                                          (5000, 1000, False), (700, 1000, True)])
def test_proposal_layer_matches_oracle(A, count, ties):
    from sln_amodal_b200 import proposal_layer
    probs, deltas, anchors = _proposal_inputs(A, 31 + A % 97, ties)
    want, aux = oracle.proposal_layer(probs, deltas, anchors, count, 0.7, return_aux=True)
    got = proposal_layer([cuda(probs).unsqueeze(0), cuda(deltas).unsqueeze(0)], count, 0.7, cuda(anchors), _Cfg())
    assert got.dim() == 3 and got.shape[0] == 1 and got.shape[2] == 4
    g = got[0].cpu().numpy()
    assert g.shape == want.shape, (g.shape, want.shape)
    # same survivors in the same order; decoded coordinates within 2 ulp (exp differs by <= 1 ulp)
    np.testing.assert_allclose(g, want, rtol=3e-7, atol=1e-7)


# --------------------------------------------------------------------------- layer codec + EDT
@pytest.mark.parametrize("num_classes", [2, 3, 5])
def test_layer_decode_bit_exact(num_classes):
    from sln_amodal_b200 import decode_layers
    labels = np.stack([synth.label_map(192, 256, n=12, seed=2024 + i, min_piece=32) for i in range(3)])
    planes, n_obj = decode_layers(labels, num_classes, n_max=20)
    planes, n_obj = planes.cpu().numpy(), n_obj.cpu().numpy()
    for b in range(3):
        want, n = oracle.layer_decode(labels[b], num_classes - 1, n_max=20)
        assert n_obj[b] == n
        assert planes[b].tobytes() == want.tobytes()
    loops = oracle.layer_decode_loops(labels[0], num_classes)
    assert np.array_equal(planes[0, :n_obj[0]].transpose(2, 3, 1, 0).astype(bool), loops)


def test_layer_decode_ragged_and_edges():
    from sln_amodal_b200 import decode_layers
    lab = synth.label_map(37, 53, n=5, seed=3, min_piece=4)
    lab[0, :5] = (1 << 0) | (1 << 1)
    lab[1, :5] = np.uint64(1 << 35)
    planes, n_obj = decode_layers(lab, 4, n_max=8)
    want, n = oracle.layer_decode(lab, 3, n_max=8)
    assert int(n_obj[0]) == n and planes[0].cpu().numpy().tobytes() == want.tobytes()
    planes, n_obj = decode_layers(np.zeros((16, 16), np.uint64), 3, n_max=4)
    assert int(n_obj[0]) == 0 and not planes.any()


def test_edt_bit_exact():
    from sln_amodal_b200 import ops
    rng = np.random.default_rng(5)
    for H, W, p in [(1, 1, 0.5), (1, 37, 0.7), (41, 1, 0.7), (37, 53, 0.9), (64, 64, 0.999), (128, 96, 0.5),
                    (70, 1100, 0.98), (33, 2100, 0.995)]:
        m = (rng.random((2, H, W)) < p).astype(np.uint8)
        m[1] = 1
        m[1].flat[rng.integers(0, H * W)] = 0
        got = ops.edt_sq_device(cuda(m)).cpu().numpy()
        for i in range(2):
            assert np.array_equal(got[i], oracle.edt_sq(m[i])), (H, W, p, i)
    full = np.ones((1, 9, 12), np.uint8)
    assert np.all(ops.edt_sq_device(cuda(full)).cpu().numpy() == (9 + 12) ** 2)


def test_edt_banded_shapes_and_field_limits():
    """The banded kernels at the edges of their contract: the tallest / widest map the packed entries allow (2048 x 1024:
    s and t up to 2047, g up to 1023), a cut last band (H % 32 != 0), a single band, one segment, and maps whose runs
    cross every band (columns of foreground from top to bottom next to far-away zeros) -- bit-exact against the oracle,
    and identical to the round-1 whole-column kernels (SLN_EDT_IMPL=legacy) on the same input."""
    import os
    from sln_amodal_b200 import ops
    rng = np.random.default_rng(91)
    cases = []
    m = np.ones((2048, 1024), np.uint8)
    m[:, 0] = 0                                              # row distances up to 1023, no zero above / below anywhere
    cases.append(m)
    m = np.ones((2048, 1024), np.uint8)
    m[2047, 1023] = 0                                        # one zero in the far corner: distances up to 2047^2 + 1023^2
    cases.append(m)
    m = (rng.random((2048, 1024)) < 0.9995).astype(np.uint8)
    cases.append(m)
    yy, xx = np.mgrid[0:2048, 0:1024]
    cases.append((((yy - 1000) / 990.0) ** 2 + ((xx - 500) / 480.0) ** 2 <= 1.0).astype(np.uint8))
    for H, W in ((1, 32), (31, 64), (33, 32), (95, 96), (250, 1024)):
        a = (rng.random((H, W)) < 0.97).astype(np.uint8)
        b = np.ones((H, W), np.uint8)
        b[rng.integers(0, H), rng.integers(0, W)] = 0
        cases += [a, b, np.ones((H, W), np.uint8)]
    for m in cases:
        got = ops.edt_sq_device(cuda(m[None])).cpu().numpy()[0]
        assert np.array_equal(got, oracle.edt_sq(m)), m.shape
        os.environ["SLN_EDT_IMPL"] = "legacy"
        try:
            old = ops.edt_sq_device(cuda(m[None])).cpu().numpy()[0]
        finally:
            os.environ.pop("SLN_EDT_IMPL", None)
        assert np.array_equal(got, old), m.shape


@pytest.mark.parametrize("L", [1, 2, 4])
def test_edt_config4_planes_bit_exact(L):
    """BASELINE config 4 on the 1024^2 path the bench times: the planes of the four distinct label maps of the bench
    workload (20 instances, L visibility layers: 80 L planes) plus the hard shapes -- an all-foreground plane, a
    full-height and a full-width blob (the longest envelope chains), a one-pixel hole, salt-and-pepper noise, stripes --
    every one bit-exact against the oracle."""
    from sln_amodal_b200 import ops
    n_inst = 20
    labels = np.stack([synth.label_map(1024, 1024, n=n_inst, seed=2024 + i) for i in range(4)])
    planes, n_obj = ops.layer_decode_device(cuda(labels.view(np.int64)), L, n_inst)          # [4, 20, L, 1024, 1024]
    rng = np.random.default_rng(40 + L)
    hard = np.zeros((8, 1024, 1024), np.uint8)
    hard[0] = 1                                             # all foreground: the (H + W)^2 sentinel
    hard[1, :, 300:620] = 1                                 # full-height blob
    hard[2, 200:777, :] = 1                                 # full-width blob
    hard[3] = 1
    hard[3, 511, 512] = 0                                   # one hole: distances up to the far corners
    hard[4] = (rng.random((1024, 1024)) < 0.97).astype(np.uint8)
    hard[5] = (rng.random((1024, 1024)) < 0.5).astype(np.uint8)
    hard[6, :, ::37] = 1
    hard[6, ::53, :] = 1                                    # thin stripes both ways
    yy, xx = np.mgrid[0:1024, 0:1024]
    hard[7] = (((yy - 500) / 480.0) ** 2 + ((xx - 530) / 470.0) ** 2 <= 1.0).astype(np.uint8)   # one huge ellipse
    allp = torch.cat([planes.reshape(-1, 1024, 1024), cuda(hard)], 0).contiguous()
    dist = ops.edt_sq_device(allp).cpu().numpy()
    host = allp.cpu().numpy()
    checked = 0
    for i in range(host.shape[0]):
        if i < host.shape[0] - 8 and not host[i].any():
            assert not dist[i].any()                        # empty plane (object absent from that layer)
            continue
        assert np.array_equal(dist[i], oracle.edt_sq(host[i])), f"plane {i}"
        checked += 1
    assert checked >= 32


def test_sem_dist_targets_end_to_end():
    from sln_amodal_b200 import sem_dist_targets
    labels = np.stack([synth.label_map(256, 256, n=8, seed=50 + i, min_piece=32) for i in range(2)])
    out = sem_dist_targets(labels, 3, n_max=8)
    planes = out["layers"].cpu().numpy()
    dist = out["dist_sq"].cpu().numpy()
    for b in range(2):
        want, _ = oracle.layer_decode(labels[b], 2, n_max=8)
        assert planes[b].tobytes() == want.tobytes()
        for i in range(8):
            for l in range(2):
                assert np.array_equal(dist[b, i, l], oracle.edt_sq(want[i, l]))


# --------------------------------------------------------------------------- size-independent properties at full size
def test_full_size_properties():
    """BASELINE config sizes, checked through properties instead of the (slow) oracle."""
    from sln_amodal_b200 import ops
    torch.manual_seed(0)
    B, C, H = 2, 256, 256
    img = torch.randn(B, C, H, H, device=dev()).contiguous(memory_format=torch.channels_last)
    # identity crop: box (0,0,1,1) at pool == map size reproduces the map exactly
    ident = ops.crop_and_resize_forward(img, torch.tensor([[0., 0., 1., 1.]] * B, device=dev()),
                                        torch.arange(B, device=dev(), dtype=torch.int32), H, H)
    assert torch.equal(ident, img)
    # linearity of forward; adjointness <crop(x), g> == <x, crop^T(g)>
    boxes = cuda(synth.roi_boxes(1000, seed=1))
    ind = torch.randint(0, B, (1000,), device=dev(), dtype=torch.int32)
    y = ops.crop_and_resize_forward(img, boxes, ind, 7, 7)
    g = torch.randn_like(y)
    gx = ops.crop_and_resize_backward(g, boxes, ind, img.shape)
    lhs = (y.double() * g.double()).sum().item()
    rhs = (img.double() * gx.double()).sum().item()
    assert abs(lhs - rhs) <= 1e-4 * max(abs(lhs), 1.0)
    # NMS idempotence at 12k: running NMS on the survivors keeps all of them
    n = 12000
    dets = cuda(np.concatenate([synth.nms_boxes(n, seed=3), synth.nms_scores(n, seed=4)[:, None]], 1))
    keep, num = ops.nms_device(dets, 0.7)
    k = int(num.item())
    keep2, num2 = ops.nms_device(dets[keep[:k]], 0.7)
    assert int(num2.item()) == k and torch.equal(keep2[:k], torch.arange(k, device=dev()))
    # EDT at 1024^2: zero exactly on zero pixels, 1-Lipschitz-ish in sqrt, equals oracle on one map
    lab = synth.label_map(1024, 1024, n=6, seed=11)
    m = ((lab & np.uint64(1)) != 0).astype(np.uint8)
    d = ops.edt_sq_device(cuda(m)).cpu().numpy()
    assert np.array_equal(d == 0, m == 0)
    assert np.array_equal(d, oracle.edt_sq(m))


def _ref_or_oracle():
    """The reference's own C (oracle/_ref, compiled from /root/reference in place) when it travelled to this box, else the
    restatement that tests/test_oracle_pin.py holds bit-identical to it."""
    if oracle.ref_available():
        return oracle.ref_crop_and_resize_fwd, oracle.ref_crop_and_resize_bwd, "reference C (oracle/_ref)"
    return oracle.crop_and_resize_fwd, oracle.crop_and_resize_bwd, "oracle restatement"


@pytest.mark.parametrize("pool", [7, 14, 16])
def test_config2_full_size_values_vs_reference_c(pool):
    """BASELINE config 2 at FULL size -- 8 images, C = 256, P2..P5 = 256^2 .. 32^2, 8 x 1000 ROIs assigned to levels by the
    FPN formula -- compared VALUE BY VALUE with the reference's own crop_and_resize.c: forward bit-exact; backward (all
    levels in one call, the bulk-async kernel) bit-exact in exact mode and within 1e-5 (north star) in the default mode."""
    from sln_amodal_b200 import ops
    ref_fwd, ref_bwd, _ = _ref_or_oracle()
    B, C, per = 8, 256, 1000
    sides = (256, 128, 64, 32)
    n = B * per
    boxes = synth.roi_boxes(n, seed=4321, outside_frac=0.05)
    level = (synth.fpn_level(boxes) - 2).astype(np.int32)
    ind = np.repeat(np.arange(B, dtype=np.int32), per)
    gen = torch.Generator(device="cpu").manual_seed(1234 + pool)
    maps = [torch.randn((B, C, s, s), generator=gen) for s in sides]
    tm = [m.to(dev()).contiguous(memory_format=torch.channels_last) for m in maps]
    tb, ti, tl = cuda(boxes), cuda(ind), cuda(level)
    got_f = ops.pyramid_crop_forward(tm, tb, ti, tl, pool, pool, 0.0).contiguous().cpu().numpy()
    g = torch.randn((n, C, pool, pool), generator=gen)
    gt = g.to(dev()).contiguous(memory_format=torch.channels_last)
    sizes = [tuple(m.shape) for m in maps]
    got_exact = [o.contiguous().cpu().numpy() for o in ops.pyramid_crop_backward(gt, tb, ti, tl, sizes, exact=True)]
    got_fast = [o.contiguous().cpu().numpy() for o in ops.pyramid_crop_backward(gt, tb, ti, tl, sizes, exact=False)]
    gn = g.numpy()
    for l, m in enumerate(maps):
        ix = np.nonzero(level == l)[0]
        assert ix.size > 500                                       # every level is populated
        want_f = ref_fwd(m.numpy(), boxes[ix], ind[ix], pool, pool, 0.0)
        assert got_f[ix].tobytes() == want_f.tobytes(), f"forward differs on level {l}"
        want_b = ref_bwd(np.ascontiguousarray(gn[ix]), boxes[ix], ind[ix], tuple(m.shape))
        assert got_exact[l].tobytes() == want_b.tobytes(), f"exact backward differs on level {l}"
        assert_close_rel(got_fast[l], want_b)
        assert_close_rel(got_fast[l], want_b, rtol=2e-6)


def test_config2_contention_4000_rois_per_image_vs_reference_c():
    """The 4000-ROIs-per-image contention case: every ROI of an image inside one small window of a 64^2 map, so a few
    hundred pixels each collect thousands of terms.  Values against the reference's crop_and_resize.c."""
    from sln_amodal_b200 import ops
    _, ref_bwd, _ = _ref_or_oracle()
    B, C, H, per, pool = 2, 256, 64, 4000, 14
    n = B * per
    boxes = synth.roi_boxes(n, seed=99, window=(0.5, 0.5, 0.06))
    ind = np.repeat(np.arange(B, dtype=np.int32), per)
    gen = torch.Generator(device="cpu").manual_seed(7)
    g = torch.randn((n, C, pool, pool), generator=gen)
    want = ref_bwd(g.numpy(), boxes, ind, (B, C, H, H))
    gt = g.to(dev()).contiguous(memory_format=torch.channels_last)
    got = ops.crop_and_resize_backward(gt, cuda(boxes), cuda(ind), (B, C, H, H), exact=True).contiguous().cpu().numpy()
    assert got.tobytes() == want.tobytes()
    got = ops.crop_and_resize_backward(gt, cuda(boxes), cuda(ind), (B, C, H, H), exact=False).contiguous().cpu().numpy()
    assert_close_rel(got, want)


@pytest.mark.parametrize("C,H,W,N,ph,pw", [(256, 40, 40, 200, 7, 7), (128, 50, 70, 150, 32, 32), (68, 21, 37, 120, 9, 20),
                                           (512, 24, 24, 60, 14, 14)])
@pytest.mark.parametrize("misaligned", [False, True], ids=["bulk-async", "strip-vec1"])
def test_backward_kernel_forms_agree(misaligned, C, H, W, N, ph, pw):
    """Both backward forms produce the oracle's bits in exact mode, also for flipped / degenerate boxes, ragged maps and
    crops that need several stages per sample row: aligned grads take the bulk-async kernel, channels_last-dense grads
    4 bytes off a 16-byte boundary the strip kernel with scalar loads."""
    from sln_amodal_b200 import ops
    rng = np.random.default_rng(5 + N)
    B = 2
    boxes = synth.roi_boxes(N, seed=N, outside_frac=0.2, degenerate_frac=0.1)
    boxes[::7] = boxes[::7][:, [2, 1, 0, 3]]                   # y-flipped
    boxes[::11] = boxes[::11][:, [0, 3, 2, 1]]                 # x-flipped
    ind = rng.integers(0, B, N).astype(np.int32)
    g = rng.standard_normal((N, C, ph, pw), dtype=np.float32)
    want = oracle.crop_and_resize_bwd(g, boxes, ind, (B, C, H, W))
    if misaligned:
        nhwc = torch.empty(g.size + 1, dtype=torch.float32, device=dev())[1:].view(N, ph, pw, C)
        nhwc.copy_(torch.from_numpy(np.ascontiguousarray(g.transpose(0, 2, 3, 1))))
        gt = nhwc.permute(0, 3, 1, 2)
        assert gt.is_contiguous(memory_format=torch.channels_last) and gt.data_ptr() % 16 == 4
    else:
        gt = cuda(g).contiguous(memory_format=torch.channels_last)
    got = ops.crop_and_resize_backward(gt, cuda(boxes), cuda(ind), (B, C, H, W), exact=True).contiguous().cpu().numpy()
    assert got.tobytes() == want.tobytes()
    got = ops.crop_and_resize_backward(gt, cuda(boxes), cuda(ind), (B, C, H, W), exact=False).contiguous().cpu().numpy()
    assert_close_rel(got, want, rtol=2e-6)


@pytest.mark.parametrize("pool", [7, 14])
def test_backward_planned_ahead_is_bit_identical(pool):
    """SLN_BWD_PLAN_ONLY + SLN_BWD_PLANNED: the ROI lists built ahead on a side stream give the same bits as the plain
    call (exact and default mode), a plan can be replayed, a plan for other boxes is ignored, and the autograd path
    (which plans beside the forward) matches the path that plans inside the backward."""
    from sln_amodal_b200 import ops, pyramid, pyramid_roi_align
    rng = np.random.default_rng(pool)
    B, C, N = 2, 256, 700
    sides = (64, 32, 16, 8)
    sizes = [(B, C, s, s) for s in sides]
    boxes = synth.roi_boxes(N, seed=31 + pool, outside_frac=0.1, degenerate_frac=0.05)
    ind = rng.integers(0, B, N).astype(np.int32)
    level = rng.integers(0, 4, N).astype(np.int32)
    g = cuda(rng.standard_normal((N, C, pool, pool), dtype=np.float32)).contiguous(memory_format=torch.channels_last)
    tb, ti, tl = cuda(boxes), cuda(ind), cuda(level)
    for exact in (True, False):
        plain = ops.pyramid_crop_backward(g, tb, ti, tl, sizes, exact=exact)
        plan = ops.pyramid_crop_backward_plan(tb, ti, tl, sizes, C, pool, pool)
        for _ in range(2):                                  # a plan is reusable
            got = ops.pyramid_crop_backward(g, tb, ti, tl, sizes, exact=exact, plan=plan)
            assert all(torch.equal(a, b) for a, b in zip(plain, got))
        other = cuda(synth.roi_boxes(N, seed=5))
        want_other = ops.pyramid_crop_backward(g, other, ti, tl, sizes, exact=exact)
        got_other = ops.pyramid_crop_backward(g, other, ti, tl, sizes, exact=exact, plan=plan)   # key mismatch: plain call
        assert all(torch.equal(a, b) for a, b in zip(want_other, got_other))
    # a plan is keyed on the CALLER's tensors: converted copies (int64 box_ind) still match, an in-place change does not
    from sln_amodal_b200 import _lib
    ti64 = ti.to(torch.int64)
    plan64 = ops.pyramid_crop_backward_plan(tb, ti64, tl, sizes, C, pool, pool)
    l0 = _lib.launches()
    got = ops.pyramid_crop_backward(g, tb, ti64, tl, sizes, plan=plan64)
    assert _lib.launches() - l0 == 2                                   # republish + main kernel: the plan was taken
    assert all(torch.equal(a, b) for a, b in zip(plain, got))
    ti64.add_(0)                                                       # version bump
    l0 = _lib.launches()
    got = ops.pyramid_crop_backward(g, tb, ti64, tl, sizes, plan=plan64)
    assert _lib.launches() - l0 == 4                                   # plan ignored: three prep launches + main kernel
    assert all(torch.equal(a, b) for a, b in zip(plain, got))
    # shapes that do not take the bulk-async kernel (ragged channel count) ignore the plan flags; an empty ROI set plans nothing
    sizes6 = [(B, 6, s, s) for s in sides]
    g6 = cuda(rng.standard_normal((N, 6, pool, pool), dtype=np.float32))
    want6 = ops.pyramid_crop_backward(g6, tb, ti, tl, sizes6, exact=True)
    got6 = ops.pyramid_crop_backward(g6, tb, ti, tl, sizes6, exact=True, plan=ops.pyramid_crop_backward_plan(tb, ti, tl, sizes6, 6, pool, pool))
    assert all(torch.equal(a, b) for a, b in zip(want6, got6))
    e_b, e_i = tb[:0], ti[:0]
    plan0 = ops.pyramid_crop_backward_plan(e_b, e_i, tl[:0], sizes, C, pool, pool)
    got0 = ops.pyramid_crop_backward(g[:0], e_b, e_i, tl[:0], sizes, plan=plan0)
    assert all(float(o.abs().max()) == 0.0 for o in got0)
    # exact mode against the oracle, level by level
    got = ops.pyramid_crop_backward(g, tb, ti, tl, sizes, exact=True, plan=ops.pyramid_crop_backward_plan(tb, ti, tl, sizes, C, pool, pool))
    gn = g.contiguous().cpu().numpy()
    for l, s in enumerate(sides):
        ix = np.nonzero(level == l)[0]
        want = oracle.crop_and_resize_bwd(gn[ix], boxes[ix], ind[ix], (B, C, s, s))
        assert got[l].contiguous().cpu().numpy().tobytes() == want.tobytes()
    # the autograd operator: planning beside the forward vs inside the backward
    maps_np = [rng.standard_normal((1, 64, s, s), dtype=np.float32) for s in sides]
    roi = cuda(synth.roi_boxes(300, seed=3)).unsqueeze(0)
    res = []
    for flag in (True, False):
        pyramid.PLAN_BACKWARD_IN_FORWARD = flag
        try:
            tm = [cuda(m).contiguous(memory_format=torch.channels_last).requires_grad_(True) for m in maps_np]
            out = pyramid_roi_align([roi] + tm, pool, (256, 256, 3))
            (out * out).sum().backward()
            res.append([t.grad.clone() for t in tm])
        finally:
            pyramid.PLAN_BACKWARD_IN_FORWARD = True
    assert all(torch.equal(a, b) for a, b in zip(*res))


# --------------------------------------------------------------------------- SURVEY 8(f)-2: extract_bboxes
def _extract_bboxes_reference(mask):
    """utils.py:28-54 restated in numpy (same RNG draws)."""
    boxes = np.zeros([mask.shape[-1], 4], dtype=np.int32)
    for i in range(mask.shape[-1]):
        m = mask[:, :, i]
        hz = np.where(np.any(m, axis=0))[0]
        vt = np.where(np.any(m, axis=1))[0]
        if hz.shape[0]:
            x1, x2 = hz[[0, -1]]
            y1, y2 = vt[[0, -1]]
            x2 += 1
            y2 += 1
        else:
            x1, x2, y1, y2 = 0, 0, 0, 0
        box = np.array([y1, x1, y2, x2]) + (np.random.rand(4) * 2 - 1) * (y2 - y1, x2 - x1, y2 - y1, x2 - x1) / 15
        box[box < 0] = 0
        boxes[i] = box
    return boxes.astype(np.int32)


@pytest.mark.parametrize("H,W", [(1024, 1024), (96, 130), (33, 17)])
def test_extract_bboxes_matches_the_numpy_rule(H, W):
    from sln_amodal_b200 import extract_bboxes, ops
    rng = np.random.default_rng(H + W)
    n = 9
    mask = np.zeros((H, W, n), np.uint8)
    for i in range(n - 2):
        y1, x1 = rng.integers(0, H - 3), rng.integers(0, W - 3)
        y2, x2 = rng.integers(y1 + 1, H + 1), rng.integers(x1 + 1, W + 1)
        mask[y1:y2, x1:x2, i] = rng.random((y2 - y1, x2 - x1)) < 0.3
    mask[H - 1, W - 1, n - 2] = 1                      # a single pixel in the last corner; plane n-1 stays empty
    planes = cuda(np.ascontiguousarray(np.moveaxis(mask, -1, 0)))
    tight = ops.plane_bboxes_device(planes).cpu().numpy()
    for i in range(n):
        ys, xs = np.nonzero(mask[:, :, i])
        want = (ys.min(), xs.min(), ys.max() + 1, xs.max() + 1) if ys.size else (0, 0, 0, 0)
        assert tuple(tight[i]) == want
    np.random.seed(3)
    want = _extract_bboxes_reference(mask)
    np.random.seed(3)
    assert np.array_equal(extract_bboxes(mask), want)
    np.random.seed(3)
    assert np.array_equal(extract_bboxes(planes), want)


# --------------------------------------------------------------------------- SURVEY 8(f)-3: COCO RLE
def test_rle_encode_matches_maskapi():
    """Device run-length encoding against the reference's own rleEncode / rleToString (cocoapi/common/maskApi.c compiled
    into oracle/_ref) where it is present, and against the oracle's restatement everywhere."""
    from sln_amodal_b200 import rle
    rng = np.random.default_rng(5)
    for h, w in ((1024, 1024), (37, 53), (5, 3), (1, 1)):
        n = 7
        masks = np.zeros((n, h, w), np.uint8)
        masks[0] = rng.random((h, w)) < 0.5                      # noise: ~a/2 runs (needs the capacity retry at 1024^2)
        masks[2] = 1                                             # all ones: [0, a]
        masks[3, : max(h // 3, 1)] = 1                           # starts with a one
        yy, xx = np.mgrid[0:h, 0:w]
        masks[4] = ((yy - h / 2) ** 2 + (xx - w / 2) ** 2) < (min(h, w) / 3) ** 2
        masks[5] = masks[4] * 3                                  # non-binary values: a change is any difference
        masks[6, h - 1, w - 1] = 1                               # last pixel only
        got = rle.encode(cuda(masks))
        cols = np.ascontiguousarray(masks.transpose(0, 2, 1)).reshape(n, h * w)
        ref = oracle.ref_rle_encode(cols, h, w) if oracle.ref_mask_available() else None
        for i in range(n):
            want_c = oracle.rle_encode(cols[i])
            assert got[i]["size"] == [h, w]
            assert got[i]["counts"] == oracle.rle_to_string(want_c), (h, w, i)
            if ref is not None:
                assert np.array_equal(ref[i][0], want_c) and got[i]["counts"] == ref[i][1]
        hwn = np.ascontiguousarray(masks.transpose(1, 2, 0))      # pycocotools' [h, w, n] convention
        assert [r["counts"] for r in rle.encode(hwn)] == [r["counts"] for r in got]


def test_resize_layer_matches_scipy_zoom():
    """utils.resize_layer = scipy.ndimage.zoom(mask, [sy, sx, 1, 1], order=0) (utils.py:358-362) and np.fliplr, on the
    device, against scipy itself -- incl. a size pair whose last column scipy zero-fills."""
    import scipy.ndimage as ndi
    from sln_amodal_b200 import resize_layer, resize_layer_device
    rng = np.random.default_rng(9)
    for (h, w), scale in (((328, 414), (1.8358701484000286, 0.49965678675982783)), ((480, 640), (1024 / 480, 1024 / 640)),
                          ((97, 61), (0.5, 2.25)), ((64, 64), (1.0, 1.0))):
        mask = (rng.random((h, w, 3, 2)) < 0.4).astype(np.uint8)            # reference layout [H, W, n, L]
        want = ndi.zoom(mask, zoom=[scale[0], scale[1], 1, 1], order=0)
        assert np.array_equal(resize_layer(mask, scale, None), want)
        planes = cuda(np.ascontiguousarray(np.moveaxis(mask, (0, 1), (-2, -1))))
        got = resize_layer_device(planes, scale, flip=True).cpu().numpy()
        assert np.array_equal(np.moveaxis(got, (-2, -1), (0, 1)), np.fliplr(want))


# --------------------------------------------------------------------------- unmold_mask (8(f)-3)
def _unmold_cases(rng, n, H, W, mh=28, mw=28):
    masks = rng.random((n, mh, mw)).astype(np.float32) ** 2
    masks[0] = 0.3                                                          # constant mask (cscale == 0)
    boxes = np.zeros((n, 4), np.int32)
    for i in range(n):
        bh = int(rng.integers(1, H + 1)) if i % 4 else int(rng.integers(1, min(mh, H)))     # every 4th: downscale
        bw = int(rng.integers(1, W + 1)) if i % 3 else int(rng.integers(1, min(mw, W)))
        y1 = int(rng.integers(0, H - bh + 1))
        x1 = int(rng.integers(0, W - bw + 1))
        boxes[i] = (y1, x1, y1 + bh, x1 + bw)
    boxes[1] = (0, 0, H, W)                                                 # whole image
    boxes[2] = (5, 7, 5, 40)                                                # empty: pastes nothing
    return masks, boxes


@pytest.mark.parametrize("H,W,mh,mw", [(256, 320, 28, 28), (130, 131, 28, 28), (192, 160, 14, 33)])
def test_unmold_masks_match_oracle(H, W, mh, mw):
    """sln_unmold_masks against the oracle's restatement of scipy bytescale + Pillow's bilinear resample (pinned to
    Pillow itself on the CPU): bit-identical planes, vector (W % 16 == 0) and byte paths."""
    from sln_amodal_b200 import unmold
    rng = np.random.default_rng(H + W)
    masks, boxes = _unmold_cases(rng, 24, H, W, mh, mw)
    got = unmold.unmold_masks(cuda(masks), cuda(boxes), (H, W, 3)).cpu().numpy()
    for i in range(masks.shape[0]):
        want = oracle.unmold_mask(masks[i], boxes[i], (H, W, 3))
        assert np.array_equal(got[i], want), (i, boxes[i].tolist(), int((got[i] != want).sum()))
    one = unmold.unmold_mask(masks[3][None], boxes[3], (H, W, 3))
    assert isinstance(one, np.ndarray) and np.array_equal(one, got[3])          # numpy like the reference's; device=True keeps it
    assert np.array_equal(unmold.unmold_mask(masks[3], boxes[3], (H, W, 3), device=True).cpu().numpy(), got[3])
    with pytest.raises(ValueError):                                            # a box past the border: the reference's paste raises
        unmold.unmold_mask(masks[3], [0, 0, H + 1, 5], (H, W, 3))


def test_unmold_detections_full_size_and_rle():
    """model.py:747-806 end to end at 1024^2: detections + class masks -> boxes / pasted planes -> COCO RLE strings,
    against the oracle (same numpy box arithmetic, restated resize) and the restated maskApi coder."""
    from sln_amodal_b200 import rle, unmold
    rng = np.random.default_rng(11)
    H = W = 1024
    N, pad = 12, 4
    det = np.zeros((N + pad, 6), np.float32)
    yx = rng.uniform(0, 700, (N, 2)).astype(np.float32)
    det[:N, 0:2] = yx
    det[:N, 2:4] = yx + rng.uniform(2, 320, (N, 2)).astype(np.float32)
    det[:N, 4] = rng.integers(1, 5, N)
    det[:N, 5] = rng.random(N)
    det[3, 2] = det[3, 0]                                                   # zero-area detection: filtered out
    mm = rng.random((N + pad, 28, 28, 2)).astype(np.float32)
    window = np.array([0, 0, 1024, 1024])
    boxes, cls, scores, planes = unmold.unmold_detections(det, mm, (H, W, 3), window, return_device_planes=True)
    assert boxes.shape == (N - 1, 4) and planes.shape == (N - 1, H, W) and np.all(cls == 1)
    keep = [i for i in range(N) if i != 3]
    got = planes.cpu().numpy()
    for j, i in enumerate(keep):
        want = oracle.unmold_mask(mm[i, :, :, 1], boxes[j], (H, W, 3))
        assert np.array_equal(got[j], want), (i, boxes[j].tolist())
    enc = rle.encode(planes)
    for j in range(len(keep)):
        col = np.ascontiguousarray(got[j].T).reshape(-1)
        assert enc[j]["counts"] == oracle.rle_to_string(oracle.rle_encode(col))
    b2, c2, s2, hwn = unmold.unmold_detections(det, mm, (H, W, 3), window)
    assert hwn.shape == (H, W, N - 1) and np.array_equal(hwn[:, :, 0], got[0])


# --------------------------------------------------------------------------- RPN re-layout (8(f)-4)
def _ref_rpn_expr(cls_maps, box_maps):
    """RPN.forward's re-layout (modal/modals.py:394-410) + the concatenation of model.py:553-563, as torch ops."""
    lg = [c.permute(0, 2, 3, 1).contiguous().view(c.size(0), -1, 2) for c in cls_maps]
    bx = [b.permute(0, 2, 3, 1).contiguous().view(b.size(0), -1, 4) for b in box_maps]
    return torch.cat(lg, 1), torch.cat([torch.softmax(x, dim=2) for x in lg], 1), torch.cat(bx, 1)


def test_rpn_pack_matches_reference_module_fixture():
    """sln_rpn_pack on the conv outputs captured from the reference's RPN module against what the module + the
    concatenation of MaskRCNN.predict returned (tests/golden/rpn_pack.npz): logits and deltas bit for bit; softmax within
    1e-6 relative of the reference's CPU kernel (the only floating-point step; tolerance per BASELINE north_star 1e-5)."""
    import os
    from sln_amodal_b200 import rpn
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rpn_pack.npz"))
    cls_maps = [cuda(g["cls_%d" % l]) for l in range(3)]
    box_maps = [cuda(g["box_%d" % l]) for l in range(3)]
    logits, probs, bbox = rpn.rpn_pack(cls_maps, box_maps)
    assert np.array_equal(logits.cpu().numpy(), g["rpn_class_logits"])
    assert np.array_equal(bbox.cpu().numpy(), g["rpn_bbox"])
    assert np.allclose(probs.cpu().numpy(), g["rpn_class"], rtol=1e-6, atol=0)
    # channels_last conv outputs take the NHWC branch: same result
    cl = [t.contiguous(memory_format=torch.channels_last) for t in cls_maps]
    bl = [t.contiguous(memory_format=torch.channels_last) for t in box_maps]
    l2, p2, b2 = rpn.rpn_pack(cl, bl)
    assert torch.equal(l2, logits) and torch.equal(p2, probs) and torch.equal(b2, bbox)


@pytest.mark.parametrize("a", [3, 2])
def test_rpn_pack_full_size_and_backward(a):
    """BASELINE shape (five levels of a 1024^2 image, 261 888 anchors at a = 3): forward against the torch expression of
    the reference on the same device (copies bit-exact, softmax <= 1e-6 relative), oracle on one level, and the backward
    launch against autograd through that expression."""
    from sln_amodal_b200 import rpn
    torch.manual_seed(5)
    sizes = (256, 128, 64, 32, 16)
    cls_maps = [torch.randn(1, 2 * a, s, s, device=dev()) * 4 for s in sizes]
    box_maps = [torch.randn(1, 4 * a, s, s, device=dev()) for s in sizes]
    c1 = [t.clone().requires_grad_(True) for t in cls_maps]
    b1 = [t.clone().requires_grad_(True) for t in box_maps]
    c2 = [t.clone().requires_grad_(True) for t in cls_maps]
    b2 = [t.clone().requires_grad_(True) for t in box_maps]
    logits, probs, bbox = rpn.rpn_pack(c1, b1)
    rl, rp, rb = _ref_rpn_expr(c2, b2)
    assert logits.shape == (1, a * 87296, 2) and torch.equal(logits, rl) and torch.equal(bbox, rb)
    assert torch.allclose(probs, rp, rtol=1e-6, atol=0)
    ol, op, ob = oracle.rpn_pack([cls_maps[4].cpu().numpy()], [box_maps[4].cpu().numpy()])
    n4 = a * 256
    assert np.array_equal(logits.detach()[:, -n4:].cpu().numpy(), ol) and np.array_equal(bbox.detach()[:, -n4:].cpu().numpy(), ob)
    assert np.allclose(probs.detach()[:, -n4:].cpu().numpy(), op, rtol=1e-6, atol=0)
    wl, wb = torch.randn_like(rl), torch.randn_like(rb)
    ((logits * wl).sum() + (bbox * wb).sum()).backward()
    ((rl * wl).sum() + (rb * wb).sum()).backward()
    for x, y in zip(c1 + b1, c2 + b2):
        assert torch.equal(x.grad, y.grad)
    assert not probs.requires_grad


# --------------------------------------------------------------------------- resize_image (8(f)-2)
@pytest.mark.parametrize("h,w,H2,W2", [(480, 640, 1024, 1024), (1440, 1920, 1024, 1024), (37, 53, 64, 80), (300, 20, 7, 33)])
def test_resize_image_matches_oracle(h, w, H2, W2):
    """sln_resize_image_u8 against the oracle's per-band restatement of Pillow's bilinear resample (pinned to Pillow on
    the CPU): COCOA- and D2SA-sized RGB images squashed to 1024^2 like utils.resize_image does, plus odd shapes."""
    from sln_amodal_b200 import targets
    rng = np.random.default_rng(h + w)
    img = rng.integers(0, 256, (h, w, 3)).astype(np.uint8)
    got = targets.resize_image_device(img, (H2, W2)).cpu().numpy()
    want = oracle.resize_image(img, (H2, W2))
    try:
        assert np.array_equal(want, oracle.resize_image_pil(img, (H2, W2)))       # the real library, when it is installed
    except ImportError:
        pass
    assert got.shape == (H2, W2, 3) and np.array_equal(got, want)
    if h == 480:
        out, window, scale, padding = targets.resize_image(img, max_dim=1024)
        assert window == (0, 0, 1024, 1024) and scale == (1024 / 480, 1024 / 640)
        assert isinstance(out, np.ndarray) and out.dtype == np.uint8 and np.array_equal(out, want)   # numpy, like utils.resize_image
        assert np.array_equal(targets.resize_image(img, max_dim=1024, device=True)[0].cpu().numpy(), want)
        gray = targets.resize_image_device(img[:, :, 0].copy(), (H2, W2)).cpu().numpy()
        assert np.array_equal(gray, want[:, :, 0])


def test_unmold_and_resize_match_reference_fixtures():
    """The device path against what the reference's own MaskRCNN.unmold_detections and utils.resize_image returned
    (tests/golden/unmold_detections.npz, resize_image.npz; see make_golden_unmold.py)."""
    import os
    from sln_amodal_b200 import targets, unmold
    gd = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    g = np.load(os.path.join(gd, "unmold_detections.npz"))
    boxes, class_ids, scores, masks = unmold.unmold_detections(g["detections"], g["mrcnn_mask"], tuple(int(v) for v in g["image_shape"]),
                                                               g["window"])
    assert np.array_equal(boxes, g["boxes"]) and np.array_equal(class_ids, g["class_ids"]) and np.array_equal(scores, g["scores"])
    assert masks.shape == g["masks"].shape and np.array_equal(masks.astype(np.uint8), g["masks"])
    r = np.load(os.path.join(gd, "resize_image.npz"))
    out, window, scale, padding = targets.resize_image(r["image"], max_dim=64)
    assert np.array_equal(out, r["resized"]) and window == tuple(r["window"]) and np.allclose(scale, r["scale"])



# --------------------------------------------------------------------------- the head path replayed from a CUDA graph
class _GraphCfg:
    IMAGE_SHAPE = np.array([1024, 1024, 3])
    RPN_BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
    BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
    RPN_NMS_THRESHOLD = 0.7
    POOL_SIZE = 7
    MASK_POOL_SIZE = 14
    USE_NMS = False
    DETECTION_MIN_CONFIDENCE = 0.0
    DETECTION_NMS_THRESHOLD = 0.3
    DETECTION_MAX_INSTANCES = 100


def test_head_graph_replay_equals_the_eager_drop_ins():
    """pipeline.HeadGraph (every step padded and sync-free, captured once, one launch per image) against the same image
    through the reference-signature drop-ins with their host reads: proposals, classifier crops, detections and mask-head
    crops identical below the counts; a second image through the SAME graph (inputs refreshed in place) too."""
    from sln_amodal_b200 import pipeline, proposal_layer, pyramid_roi_align, refine_detections
    A, K, Cc = 65472, 9, 64
    cfg = _GraphCfg()
    rng = np.random.default_rng(5)
    anchors = cuda(synth.nms_boxes(A, seed=4, kind="rpn"))
    sides = (128, 64, 32, 16)

    def image(seed):
        r = np.random.default_rng(seed)
        fg = r.permutation(np.linspace(0, 1, A)).astype(np.float32)
        lg = r.standard_normal((1000, K)).astype(np.float32) * 3.0
        return {"probs": np.stack([1 - fg, fg], 1).astype(np.float32), "deltas": (r.standard_normal((A, 4)) * 0.5).astype(np.float32),
                "cls_probs": (np.exp(lg) / np.exp(lg).sum(1, keepdims=True)).astype(np.float32),
                "cls_deltas": (r.standard_normal((1000, K, 4)) * 0.3).astype(np.float32),
                "maps": [r.standard_normal((1, Cc, s_, s_), dtype=np.float32) for s_ in sides]}

    first = image(11)
    st = {k: cuda(v) for k, v in first.items() if k != "maps"}
    st["maps"] = [cuda(m).contiguous(memory_format=torch.channels_last) for m in first["maps"]]
    graph = pipeline.HeadGraph(anchors, cfg, st["maps"], st["probs"], st["deltas"], (st["cls_probs"], st["cls_deltas"]))
    for seed in (11, 12, 13):
        img = image(seed)
        for k in ("probs", "deltas", "cls_probs", "cls_deltas"):
            st[k].copy_(cuda(img[k]))
        for m, src in zip(st["maps"], img["maps"]):
            m.copy_(cuda(src))
        out = graph.replay()
        torch.cuda.synchronize()
        k = int(out["num_rois"].item())
        nd = int(out["num_detections"].item())
        rois = proposal_layer([st["probs"].unsqueeze(0).clone(), st["deltas"].unsqueeze(0).clone()], 1000, 0.7, anchors, cfg)
        assert rois.shape[1] == k and torch.equal(rois[0], out["rois"][:k]) and not out["rois"][k:].any()
        pooled = pyramid_roi_align([rois] + st["maps"], 7, cfg.IMAGE_SHAPE)
        assert torch.equal(pooled, out["pooled"][:k])
        det, keep = refine_detections(rois[0], st["cls_probs"][:k], st["cls_deltas"][:k], (0.0, 0.0, 1024.0, 1024.0), cfg)
        assert det.shape[0] == nd and torch.equal(det, out["detections"][:nd]) and not out["detections"][nd:].any()
        assert torch.equal(keep, out["keep"][:nd])
        mask_in = pyramid_roi_align([(det[:, :4] / 1024.0).unsqueeze(0)] + st["maps"], 14, cfg.IMAGE_SHAPE)
        assert torch.equal(mask_in, out["mask_pooled"][:nd])


def test_multi_head_graph_images_do_not_interact():
    """pipeline.MultiHeadGraph: three images as parallel branches of one graph; every image's outputs equal those of its
    own single-image graph (same kernels, own workspaces)."""
    from sln_amodal_b200 import pipeline
    A, K, Cc = 65472, 9, 64
    cfg = _GraphCfg()
    anchors = cuda(synth.nms_boxes(A, seed=4, kind="rpn"))
    sides = (128, 64, 32, 16)
    sets = []
    for seed in (21, 22, 23):
        r = np.random.default_rng(seed)
        fg = r.permutation(np.linspace(0, 1, A)).astype(np.float32)
        lg = r.standard_normal((1000, K)).astype(np.float32) * 3.0
        sets.append({"probs": cuda(np.stack([1 - fg, fg], 1).astype(np.float32)), "deltas": cuda((r.standard_normal((A, 4)) * 0.5).astype(np.float32)),
                     "cls": (cuda((np.exp(lg) / np.exp(lg).sum(1, keepdims=True)).astype(np.float32)),
                             cuda((r.standard_normal((1000, K, 4)) * 0.3).astype(np.float32))),
                     "maps": [cuda(r.standard_normal((1, Cc, s_, s_), dtype=np.float32)).contiguous(memory_format=torch.channels_last) for s_ in sides]})
    singles = [pipeline.HeadGraph(anchors, cfg, d["maps"], d["probs"], d["deltas"], d["cls"]) for d in sets]
    want = []
    for g in singles:
        o = g.replay()
        torch.cuda.synchronize()
        want.append({k: v.clone() for k, v in o.items()})
    multi = pipeline.MultiHeadGraph([pipeline.HeadGraph(anchors, cfg, d["maps"], d["probs"], d["deltas"], d["cls"], capture=False) for d in sets])
    for _ in range(3):
        outs = multi.replay()
    torch.cuda.synchronize()
    for o, w in zip(outs, want):
        k, nd = int(w["num_rois"].item()), int(w["num_detections"].item())
        assert int(o["num_rois"].item()) == k and int(o["num_detections"].item()) == nd
        assert torch.equal(o["rois"], w["rois"]) and torch.equal(o["pooled"][:k], w["pooled"][:k])
        assert torch.equal(o["detections"], w["detections"]) and torch.equal(o["mask_pooled"][:nd], w["mask_pooled"][:nd])


def test_head_graph_with_a_classifier_module_inside_the_capture():
    """HeadGraph with a torch module as the classifier callback (the place of the model's own head): the module runs inside
    the capture on the pooled crops; detections equal the eager sequence proposal_layer -> pyramid_roi_align -> the same
    module -> refine_detections."""
    from sln_amodal_b200 import pipeline, proposal_layer, pyramid_roi_align, refine_detections
    A, K, Cc = 65472, 5, 32
    cfg = _GraphCfg()
    torch.manual_seed(3)
    anchors = cuda(synth.nms_boxes(A, seed=4, kind="rpn"))
    r = np.random.default_rng(31)
    fg = r.permutation(np.linspace(0, 1, A)).astype(np.float32)
    probs, deltas = cuda(np.stack([1 - fg, fg], 1).astype(np.float32)), cuda((r.standard_normal((A, 4)) * 0.5).astype(np.float32))
    maps = [cuda(r.standard_normal((1, Cc, s_, s_), dtype=np.float32)).contiguous(memory_format=torch.channels_last) for s_ in (128, 64, 32, 16)]

    class Head(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.conv = torch.nn.Conv2d(Cc, 16, 7)
            self.cls = torch.nn.Linear(16, K)
            self.box = torch.nn.Linear(16, 4 * K)

        def forward(self, pooled, rois):
            x = torch.relu(self.conv(pooled)).flatten(1)
            return torch.softmax(self.cls(x), dim=1), self.box(x).view(-1, K, 4) * 0.1

    head = Head().to(dev()).eval()
    with torch.no_grad():
        graph = pipeline.HeadGraph(anchors, cfg, maps, probs, deltas, head)
        out = graph.replay()
        torch.cuda.synchronize()
        k, nd = int(out["num_rois"].item()), int(out["num_detections"].item())
        rois = proposal_layer([probs.unsqueeze(0).clone(), deltas.unsqueeze(0).clone()], 1000, 0.7, anchors, cfg)
        assert rois.shape[1] == k
        pooled = pyramid_roi_align([rois] + maps, 7, cfg.IMAGE_SHAPE)
        # the module sees the padded batch inside the graph; rows are independent, so the first k match a k-row call
        p_e, d_e = head(out["pooled"], out["rois"])
        det, keep = refine_detections(rois[0], p_e[:k], d_e[:k], (0.0, 0.0, 1024.0, 1024.0), cfg)
    assert torch.equal(pooled, out["pooled"][:k])
    assert det.shape[0] == nd and torch.equal(det, out["detections"][:nd]) and torch.equal(keep, out["keep"][:nd])
