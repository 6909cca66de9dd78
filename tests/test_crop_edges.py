"""RoIAlign kernels at the edges of their dispatch, and the input contract of the ops layer that feeds them.

test_gpu_parity.py covers the shapes the benchmark runs (C = 256, 7x7 .. 16x16 crops, four FPN levels, maps of 256^2
or smaller).  The kernels have more forms than that (csrc/crop.cu, csrc/crop_bwd_tma.cuh): this file reaches each of
them and compares it with the CPU oracle on the same seeded inputs, with the suite's bars:
    forward                 bit-exact
    backward, exact mode    bit-exact
    backward, default mode  <= 2e-6 relative, and the oracle's zero pattern.

GPU tests carry @gpu one by one: the input-contract tests at the end also run without a device, against a stub of the
library that fails when it is called.
"""
import contextlib
import ctypes
import re
from typing import NamedTuple

import numpy as np
import pytest
import torch

from oracle import oracle
from sln_amodal_b200 import synth

gpu = pytest.mark.gpu

RTOL_DEFAULT = 2e-6     # default-mode backward (fma per term) against the oracle


def dev():
    return torch.device("cuda", 0)


def cuda(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.to(dev())


def host(t):
    return t.detach().contiguous().cpu().numpy()


def assert_close_rel(got, want, rtol):
    got = np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    scale = max(np.abs(want).max(), 1e-30) if want.size else 1.0
    err = np.abs(got - want).max() / scale if want.size else 0.0
    assert err <= rtol, f"max rel err {err:.3e} > {rtol}"


def check_backward(exact, default, want, what=""):
    """exact: bit-identical to the oracle; default: within RTOL_DEFAULT and zero exactly where the oracle is zero."""
    assert exact.shape == want.shape and default.shape == want.shape, what
    assert exact.tobytes() == want.tobytes(), f"{what}: exact-mode backward differs from the oracle"
    assert_close_rel(default, want, RTOL_DEFAULT)
    differ = (default == 0) != (want == 0)
    assert not differ.any() or np.abs(default[differ]).max() < 1e-30, f"{what}: zero pattern differs from the oracle"


def edge_boxes(N, seed):
    """ROIs partly outside the image, degenerate (y1 == y2), y-flipped and x-flipped."""
    boxes = synth.roi_boxes(N, seed=seed, outside_frac=0.2, degenerate_frac=0.1)
    boxes[::7] = boxes[::7][:, [2, 1, 0, 3]]
    boxes[::11] = boxes[::11][:, [0, 3, 2, 1]]
    return boxes


# --------------------------------------------------------------------------- backward dispatch matrix
# `kernel` names the instantiation the case is meant to reach: (kernel name, template arguments) with "E" for the EXACT
# flag.  Two forms: crop_bwd_tma_kernel<NV, EXACT, FULL, STG_S, NST> (bulk-async) and crop_bwd_nhwc_kernel<VEC, NV, EXACT>
# (strip form, every shape the bulk-async kernel does not take).
class BwdCase(NamedTuple):
    C: int
    H: int
    W: int
    ph: int
    pw: int
    misaligned: bool
    kernel: tuple


def _n_rois(C, ph, pw):
    return int(np.clip(2_000_000 // (C * ph * pw), 12, 64))


# the bulk-async kernel: every channel class (one, two and three 256-channel chunks) x both stage configurations
_TMA_NV_FULL = {4: (1, 0), 124: (1, 0), 192: (2, 0), 260: (2, 0), 384: (2, 0), 516: (2, 0)}
_TMA_STAGES = {(8, 8): (16, 6), (5, 13): (32, 3), (1, 32): (16, 6), (32, 1): (16, 6), (32, 32): (32, 3)}   # ph*pw <= 64: 16x6
_STRIP_BIG_MAP = (128, 128)       # 16 x 32 strips x B = 2: 1024 >= 6 * 148, two channel vectors per lane
_STRIP_SMALL_MAP = (24, 20)

BWD_CASES = {}
for _C, (_nv, _full) in _TMA_NV_FULL.items():
    for (_ph, _pw), (_s, _k) in _TMA_STAGES.items():
        BWD_CASES[f"tma-nv{_nv}-{'full' if _full else 'part'}-stg{_s}x{_k}-C{_C}-{_ph}x{_pw}"] = BwdCase(
            _C, 37, 45, _ph, _pw, False, ("crop_bwd_tma_kernel", (_nv, "E", _full, _s, _k)))
for _ph, _pw in ((33, 33), (7, 40), (255, 1), (40, 255)):     # wider than 32 per side: strip form, C = 132 -> 33 vectors
    BWD_CASES[f"strip-vec4-nv2-C132-{_ph}x{_pw}-map128"] = BwdCase(
        132, *_STRIP_BIG_MAP, _ph, _pw, False, ("crop_bwd_nhwc_kernel", (4, 2, "E")))
    BWD_CASES[f"strip-vec4-nv1-C132-{_ph}x{_pw}-map24x20"] = BwdCase(
        132, *_STRIP_SMALL_MAP, _ph, _pw, False, ("crop_bwd_nhwc_kernel", (4, 1, "E")))
# channels_last-dense grads 4 bytes off a 16-byte boundary: the scalar (VEC1) strip form
BWD_CASES["strip-vec1-nv1-misaligned-C256-8x8"] = BwdCase(256, 40, 40, 8, 8, True, ("crop_bwd_nhwc_kernel", (1, 1, "E")))
BWD_CASES["strip-vec1-nv1-misaligned-C256-14x14"] = BwdCase(256, 40, 40, 14, 14, True, ("crop_bwd_nhwc_kernel", (1, 1, "E")))


def _bwd_inputs(case, seed):
    B = 2
    N = _n_rois(case.C, case.ph, case.pw)
    rng = np.random.default_rng(seed)
    boxes = edge_boxes(N, seed + 1)
    ind = rng.integers(0, B, N).astype(np.int32)
    g = rng.standard_normal((N, case.C, case.ph, case.pw), dtype=np.float32)
    if case.misaligned:
        buf = torch.empty(g.size + 1, dtype=torch.float32, device=dev())
        nhwc = buf[1:].view(N, case.ph, case.pw, case.C)
        nhwc.copy_(torch.from_numpy(np.ascontiguousarray(g.transpose(0, 2, 3, 1))))
        gt = nhwc.permute(0, 3, 1, 2)
        assert gt.is_contiguous(memory_format=torch.channels_last) and gt.data_ptr() % 16 == 4
    else:
        gt = cuda(g).contiguous(memory_format=torch.channels_last)
    return (B, case.C, case.H, case.W), boxes, ind, g, gt


@gpu
@pytest.mark.parametrize("cid", list(BWD_CASES))
def test_backward_dispatch_matrix(cid):
    from sln_amodal_b200 import ops
    case = BWD_CASES[cid]
    shape, boxes, ind, g, gt = _bwd_inputs(case, seed=len(cid) * 31 + case.C)
    want = oracle.crop_and_resize_bwd(g, boxes, ind, shape)
    tb, ti = cuda(boxes), cuda(ind)
    exact = host(ops.crop_and_resize_backward(gt, tb, ti, shape, exact=True))
    default = host(ops.crop_and_resize_backward(gt, tb, ti, shape, exact=False))
    check_backward(exact, default, want, cid)


def _template_args(name, kernel):
    """Template arguments of `kernel` in a demangled kernel name as ints ((int)2, (bool)0, false, ... all spellings)."""
    m = re.search(re.escape(kernel) + r"<([^<>]*)>", name)
    if m is None:
        return None
    args = []
    for a in m.group(1).split(","):
        a = re.sub(r"^\(\w+\)", "", a.strip())
        args.append({"true": 1, "false": 0}[a] if a in ("true", "false") else int(a))
    return tuple(args)


@gpu
def test_backward_dispatch_matrix_reaches_the_named_kernels():
    """Every id of the dispatch matrix runs the instantiation it names (kernel names from torch.profiler), so the matrix
    cannot silently collapse onto one path.  Each call launches one main kernel, so the main kernels in launch order
    line up with the calls."""
    from torch.profiler import ProfilerActivity, profile
    from sln_amodal_b200 import ops
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    H, W = _STRIP_BIG_MAP
    assert 2 * (H // 8) * (W // 4) >= 6 * sms, "the big strip map no longer gives enough strips for two vectors per lane"
    calls = []
    for cid, case in BWD_CASES.items():
        shape, boxes, ind, _, gt = _bwd_inputs(case, seed=7)
        for exact in (False, True):
            calls.append((cid, exact, gt, cuda(boxes), cuda(ind), shape))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _, exact, gt, tb, ti, shape in calls:
            ops.crop_and_resize_backward(gt, tb, ti, shape, exact=exact)
        torch.cuda.synchronize()
    kernels = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "crop_bwd" in e.name),
                     key=lambda e: e.time_range.start)
    if not kernels:
        pytest.skip("torch.profiler recorded no CUDA kernels on this host (CUPTI unavailable)")
    main = [e.name for e in kernels if re.search(r"crop_bwd_(tma|nhwc)_kernel<", e.name)]
    assert len(main) == len(calls), (len(main), len(calls))
    for name, (cid, exact, *_) in zip(main, calls):
        kernel, args = BWD_CASES[cid].kernel
        want = tuple(int(exact) if a == "E" else a for a in args)
        assert _template_args(name, kernel) == want, f"{cid} (exact={exact}) ran {name}"


# --------------------------------------------------------------------------- pyramid edges
PYR_SIZES = [(700, 300), (256, 256), (64, 57), (1, 57), (57, 1), (1, 1), (9, 9), (3, 300)]
PYR_EMPTY_LEVEL = 6


def _pyramid_inputs(C, pool, seed):
    B, N = 2, 240
    rng = np.random.default_rng(seed)
    maps = [rng.standard_normal((B, C, h, w), dtype=np.float32) for h, w in PYR_SIZES]
    boxes = edge_boxes(N, seed + 1)
    ind = rng.integers(0, B, N).astype(np.int32)
    level = rng.integers(0, len(PYR_SIZES) - 1, N).astype(np.int32)
    level[level >= PYR_EMPTY_LEVEL] += 1                      # no ROI on PYR_EMPTY_LEVEL
    level[[0, 5]] = -1
    level[[1, 9]] = len(PYR_SIZES)
    ind[[2, 6]] = -1
    ind[[3, 10]] = B
    g = rng.standard_normal((N, C, pool, pool), dtype=np.float32)
    valid = (level >= 0) & (level < len(PYR_SIZES)) & (ind >= 0) & (ind < B)
    return maps, boxes, ind, level, g, valid


@gpu
@pytest.mark.parametrize("C,pool", [(16, 7), (16, 14), (6, 7)], ids=["tma-small-stages", "tma-large-stages", "C6-strip"])
def test_pyramid_eight_levels_and_invalid_rows(C, pool):
    """Eight levels (maps above 256 a side, 1xW, Hx1, 1x1, one level without ROIs), level -1 / 8 and box_ind -1 / B.
    Forward: per-level values bit-exact, rows of an invalid level or image exactly zero.  Backward: per level, exact and
    default mode, with and without a plan built ahead; invalid rows contribute nothing."""
    from sln_amodal_b200 import ops
    maps, boxes, ind, level, g, valid = _pyramid_inputs(C, pool, seed=C + pool)
    tb, ti, tl = cuda(boxes), cuda(ind), cuda(level)
    ext = -3.5
    got = host(ops.pyramid_crop_forward([cuda(m).contiguous(memory_format=torch.channels_last) for m in maps],
                                        tb, ti, tl, pool, pool, ext))
    assert got[~valid].tobytes() == np.zeros_like(got[~valid]).tobytes()
    for lv, m in enumerate(maps):
        ix = np.nonzero(valid & (level == lv))[0]
        assert (ix.size == 0) == (lv == PYR_EMPTY_LEVEL)
        want = oracle.crop_and_resize_fwd(m, boxes[ix], ind[ix], pool, pool, ext)
        assert got[ix].tobytes() == want.tobytes(), f"forward, level {lv} {PYR_SIZES[lv]}"
    sizes = [m.shape for m in maps]
    gt = cuda(g).contiguous(memory_format=torch.channels_last)
    wants = []
    for lv, m in enumerate(maps):
        ix = np.nonzero(valid & (level == lv))[0]
        wants.append(oracle.crop_and_resize_bwd(g[ix], boxes[ix], ind[ix], m.shape))
    for planned in (False, True):
        res = {}
        for exact in (True, False):
            plan = ops.pyramid_crop_backward_plan(tb, ti, tl, sizes, C, pool, pool) if planned else None
            res[exact] = [host(o) for o in ops.pyramid_crop_backward(gt, tb, ti, tl, sizes, exact=exact, plan=plan)]
        for lv in range(len(maps)):
            check_backward(res[True][lv], res[False][lv], wants[lv], f"level {lv} {PYR_SIZES[lv]} planned={planned}")


def _crop_bwd_kernels(prof):
    """Short names (windows, group, fill, republish, tma, nhwc) of the crop_bwd kernels a profile recorded, sorted."""
    return sorted(re.search(r"crop_bwd_(\w+?)_kernel", e.name).group(1) for e in prof.events()
                  if e.device_type == torch.autograd.DeviceType.CUDA and "crop_bwd_" in e.name)


@gpu
@pytest.mark.parametrize("C,pool", [(6, 7), (16, 33)], ids=["C6-7x7", "C16-33x33"])
def test_planned_strip_backward_skips_the_prep_kernels(C, pool):
    """Shapes the bulk-async kernel does not take (ragged C, crops wider than 32 per side) plan ahead like the others: the
    plan call launches the three prep kernels, and the planned backward only republishes the level table and gathers."""
    from torch.profiler import ProfilerActivity, profile
    from sln_amodal_b200 import ops
    maps, boxes, ind, level, g, _ = _pyramid_inputs(C, pool, seed=C + pool)
    tb, ti, tl = cuda(boxes), cuda(ind), cuda(level)
    sizes = [m.shape for m in maps]
    gt = cuda(g).contiguous(memory_format=torch.channels_last)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof_plan:
        plan = ops.pyramid_crop_backward_plan(tb, ti, tl, sizes, C, pool, pool)
        torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof_bwd:
        ops.pyramid_crop_backward(gt, tb, ti, tl, sizes, plan=plan)
        torch.cuda.synchronize()
    plan_kernels, bwd_kernels = _crop_bwd_kernels(prof_plan), _crop_bwd_kernels(prof_bwd)
    if not plan_kernels and not bwd_kernels:
        pytest.skip("torch.profiler recorded no CUDA kernels on this host (CUPTI unavailable)")
    assert plan_kernels == ["fill", "group", "windows"], plan_kernels
    assert bwd_kernels == ["nhwc", "republish"], bwd_kernels


# --------------------------------------------------------------------------- forward size edges
@gpu
@pytest.mark.parametrize("C", [3, 4, 256])
@pytest.mark.parametrize("ph,pw", [(48, 48), (64, 64), (1, 3000), (3000, 1)])
def test_nhwc_forward_band_split(C, ph, pw):
    """Crops above 2048 samples are split across CTAs in bands of 2048 (ragged last band for 48x48, 1x3000, 3000x1), in
    the scalar (C = 3) and float4 (C = 4, 256) forms."""
    from sln_amodal_b200 import ops
    B, H, W, N = 2, 37, 53, 5
    rng = np.random.default_rng(C + ph)
    img = rng.standard_normal((B, C, H, W), dtype=np.float32)
    boxes = edge_boxes(N, C + pw)
    ind = rng.integers(0, B, N).astype(np.int32)
    t = cuda(img).contiguous(memory_format=torch.channels_last)
    got = ops.crop_and_resize_forward(t, cuda(boxes), cuda(ind), ph, pw, -2.5)
    assert got.is_contiguous(memory_format=torch.channels_last)          # the NHWC kernel wrote it
    assert host(got).tobytes() == oracle.crop_and_resize_fwd(img, boxes, ind, ph, pw, -2.5).tobytes()


@gpu
def test_nchw_forward_crop_with_large_tap_tables():
    """ph + pw = 6296: the NCHW kernel's tap tables need 50 KB of shared memory, above the 48 KB granted by default.
    C = 2 keeps the image on the NCHW kernel (a C = 1 tensor is channels_last as well and takes the NHWC kernel)."""
    from sln_amodal_b200 import ops
    ph, pw = 4096, 2200
    rng = np.random.default_rng(3)
    img = rng.standard_normal((1, 2, 19, 23), dtype=np.float32)
    boxes = np.array([[0.1, -0.2, 0.9, 1.1]], np.float32)
    ind = np.zeros(1, np.int32)
    got = ops.crop_and_resize_forward(cuda(img), cuda(boxes), cuda(ind), ph, pw, 0.5)
    assert got.is_contiguous() and not got.is_contiguous(memory_format=torch.channels_last)
    assert host(got).tobytes() == oracle.crop_and_resize_fwd(img, boxes, ind, ph, pw, 0.5).tobytes()


# --------------------------------------------------------------------------- mask targets
def _mask_targets_want(masks, assignment, boxes, mh, mw):
    """np.round of the oracle's crop of every (ROI, layer) plane; rows whose assignment is out of range stay zero."""
    L, G = masks.shape[:2]
    P = boxes.shape[0]
    want = np.zeros((P, L, mh, mw), np.float32)
    ok = np.nonzero((assignment >= 0) & (assignment < G))[0]
    for lv in range(L):
        planes = masks[lv].astype(np.float32)[:, None]
        want[ok, lv] = np.round(oracle.crop_and_resize_fwd(planes, boxes[ok], assignment[ok], mh, mw, 0.0))[:, 0]
    return want


@gpu
@pytest.mark.parametrize("L,G,H,W,mh,mw,kind", [
    (1, 1, 1024, 1024, 28, 28, "u8"), (3, 5, 1024, 1024, 1, 1, "bool"), (3, 5, 333, 517, 56, 56, "bool"),
    (3, 40, 333, 517, 32, 32, "u8"), (1, 40, 1, 64, 7, 33, "bool"), (1, 5, 1, 64, 28, 28, "u8"),
    (3, 1, 333, 517, 7, 33, "u8"), (1, 40, 333, 517, 1, 1, "bool"),
])
def test_mask_targets_match_rounded_oracle_crop(L, G, H, W, mh, mw, kind):
    from sln_amodal_b200 import ops
    rng = np.random.default_rng(L * 1000 + G + H)
    P = 60
    # blobs rather than noise: targets see edges, interiors and the background
    yy = np.arange(H, dtype=np.float32)[:, None] / max(H, 2)
    xx = np.arange(W, dtype=np.float32)[None, :] / W
    cy, cx, r = [rng.uniform(lo, hi, (L, G, 1, 1)).astype(np.float32) for lo, hi in ((0, 1), (0, 1), (0.1, 0.6))]
    masks = (yy - cy) ** 2 + (xx - cx) ** 2 < r ** 2
    masks ^= rng.random(masks.shape, dtype=np.float32) < 0.02
    boxes = edge_boxes(P, G + H)
    assignment = rng.integers(0, G, P).astype(np.int32)
    assignment[[0, 7]] = -1
    assignment[[1, 8]] = G
    want = _mask_targets_want(masks.astype(np.uint8), assignment, boxes, mh, mw)
    tm = cuda(masks) if kind == "bool" else cuda(masks.astype(np.uint8))
    got = host(ops.mask_targets_device(tm, cuda(assignment), cuda(boxes), mh, mw))
    assert got.tobytes() == want.tobytes()
    assert not got[[0, 1, 7, 8]].any()


@gpu
def test_mask_targets_round_half_to_even():
    """Samples halfway between two pixels: 0.5 rounds to 0 and 1.5 to 2 (half to even, like torch.round)."""
    from sln_amodal_b200 import ops
    masks = np.array([[[[0, 1], [0, 1]], [[1, 2], [1, 2]]]], np.uint8)        # [L=1, G=2, 2, 2]
    boxes = np.array([[0, 0, 1, 1], [0, 0, 1, 1]], np.float32)                # x samples at 0, 0.5, 1
    assignment = np.array([0, 1], np.int32)
    got = host(ops.mask_targets_device(cuda(masks), cuda(assignment), cuda(boxes), 2, 3))
    assert got.tobytes() == np.array([[[[0, 0, 1]] * 2], [[[1, 2, 2]] * 2]], np.float32).tobytes()
    assert got.tobytes() == _mask_targets_want(masks, assignment, boxes, 2, 3).tobytes()


# --------------------------------------------------------------------------- input contract
NON_F32 = [torch.bfloat16, torch.float16, torch.float64]


def _dtype_id(d):
    return str(d).replace("torch.", "")


@gpu
@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
@pytest.mark.parametrize("dtype", NON_F32, ids=_dtype_id)
def test_non_f32_images_crop_their_f32_values(dtype, layout):
    """bf16 / fp16 / fp64 images, NCHW or channels_last, through every crop entry point: the result is bit-equal to the
    call on image.float(), and the gradient arrives in the image's dtype, equal to the f32 gradient cast to it."""
    from sln_amodal_b200 import ops, pyramid_roi_align
    from sln_amodal_b200.crop_and_resize import CropAndResizeFunction
    fmt = torch.channels_last if layout == "channels_last" else torch.contiguous_format
    rng = np.random.default_rng(17)
    B, C, N, pool = 2, 64, 90, 7
    img = cuda(rng.standard_normal((B, C, 29, 33), dtype=np.float32)).to(dtype).contiguous(memory_format=fmt)
    boxes, ind = cuda(edge_boxes(N, 4)), cuda(rng.integers(0, B, N).astype(np.int32))
    w = cuda(rng.standard_normal((N, C, pool, pool), dtype=np.float32))

    ref = ops.crop_and_resize_forward(img.float(), boxes, ind, pool, pool, 1.5)
    assert torch.equal(ops.crop_and_resize_forward(img, boxes, ind, pool, pool, 1.5), ref)
    assert host(ref).tobytes() == oracle.crop_and_resize_fwd(host(img.float()), host(boxes), host(ind), pool, pool, 1.5).tobytes()

    maps = [cuda(rng.standard_normal((B, C, s, s + 3), dtype=np.float32)).to(dtype).contiguous(memory_format=fmt)
            for s in (32, 16, 8, 4)]
    level = cuda(rng.integers(0, 4, N).astype(np.int32))
    ref = ops.pyramid_crop_forward([m.float() for m in maps], boxes, ind, level, pool, pool)
    assert torch.equal(ops.pyramid_crop_forward(maps, boxes, ind, level, pool, pool), ref)

    def crop_grads(x):
        x = x.detach().requires_grad_(True)
        out = CropAndResizeFunction(pool, pool, 0)(x, boxes, ind)
        (out * w).sum().backward()
        return out.detach(), x.grad
    out, grad = crop_grads(img)
    out32, grad32 = crop_grads(img.float())
    assert torch.equal(out, out32)
    assert grad.dtype == dtype and torch.equal(grad, grad32.to(dtype))

    rois = boxes.unsqueeze(0)

    def pyramid_grads(ms):
        ms = [m[:1].detach().requires_grad_(True) for m in ms]
        out = pyramid_roi_align([rois] + ms, pool, (256, 256, 3))
        (out * w).sum().backward()
        return out.detach(), [m.grad for m in ms]
    out, grads = pyramid_grads(maps)
    out32, grads32 = pyramid_grads([m.float() for m in maps])
    assert torch.equal(out, out32)
    for gm, g32 in zip(grads, grads32):
        assert gm.dtype == dtype and torch.equal(gm, g32.to(dtype))


@gpu
def test_box_and_index_dtypes_and_strides():
    """fp64 boxes taken as a column slice of an [N,6] tensor, int64 box_ind / level, and the stride-0 gradient that
    .sum().backward() hands over: same values as the plain f32 / int32 / dense call."""
    from sln_amodal_b200 import ops, pyramid_roi_align
    from sln_amodal_b200.crop_and_resize import CropAndResizeFunction
    rng = np.random.default_rng(23)
    B, C, N, pool = 2, 32, 70, 7
    img_np = rng.standard_normal((B, C, 27, 31), dtype=np.float32)
    img = cuda(img_np).contiguous(memory_format=torch.channels_last)
    boxes_np, ind_np = edge_boxes(N, 9), rng.integers(0, B, N).astype(np.int32)
    rows = torch.zeros((N, 6), dtype=torch.float64, device=dev())
    rows[:, 1:5] = cuda(boxes_np, torch.float64)
    boxes = rows[:, 1:5]                         # fp64 column slice
    assert not boxes.is_contiguous()
    ind = cuda(ind_np, torch.int64)
    tb, ti = cuda(boxes_np), cuda(ind_np)

    got = ops.crop_and_resize_forward(img, boxes, ind, pool, pool)
    assert host(got).tobytes() == oracle.crop_and_resize_fwd(img_np, boxes_np, ind_np, pool, pool).tobytes()
    maps = [cuda(rng.standard_normal((B, C, s, s), dtype=np.float32)) for s in (24, 12)]
    lvl_np = rng.integers(0, 2, N).astype(np.int32)
    assert torch.equal(ops.pyramid_crop_forward(maps, boxes, ind, cuda(lvl_np, torch.int64), pool, pool),
                       ops.pyramid_crop_forward(maps, tb, ti, cuda(lvl_np), pool, pool))

    x = img.detach().requires_grad_(True)
    CropAndResizeFunction(pool, pool, 0)(x, boxes, ind).sum().backward()
    ones = torch.ones((N, C, pool, pool), device=dev())
    assert torch.equal(x.grad, ops.crop_and_resize_backward(ones, tb, ti, img.shape))
    want = oracle.crop_and_resize_bwd(np.ones((N, C, pool, pool), np.float32), boxes_np, ind_np, img.shape)
    assert_close_rel(host(x.grad), want, RTOL_DEFAULT)

    # pyramid_roi_align takes the level of f32 boxes from the kernel and of others from the torch expression: an f32
    # slice here, so that both calls put every ROI on the same level
    ms = [m[:1].detach().requires_grad_(True) for m in maps]
    pyramid_roi_align([rows.float()[:, 1:5].unsqueeze(0)] + ms, pool, (256, 256, 3)).sum().backward()
    ms32 = [m[:1].detach().requires_grad_(True) for m in maps]
    out = pyramid_roi_align([tb.unsqueeze(0)] + ms32, pool, (256, 256, 3))
    out.backward(torch.ones_like(out))
    for a, b in zip(ms, ms32):
        assert torch.equal(a.grad, b.grad)


def _mismatched_calls(ops, device):
    """Every call here passes an index / grads / map-size array that disagrees with the boxes: each must raise SlnError
    before anything is launched (a short array would be read out of bounds by the kernels)."""
    B, C, N, p = 2, 8, 10, 7
    f32 = dict(dtype=torch.float32, device=device)
    boxes = torch.rand((N, 4), **f32)
    ind = torch.zeros(N, dtype=torch.int32, device=device)
    lvl = torch.zeros(N, dtype=torch.int32, device=device)
    short = ind[:N - 1]
    maps = [torch.zeros((B, C, s, s), **f32).contiguous(memory_format=torch.channels_last) for s in (16, 8)]
    sizes = [tuple(m.shape) for m in maps]
    grads = torch.zeros((N, C, p, p), **f32).contiguous(memory_format=torch.channels_last)
    masks = torch.zeros((1, 3, 16, 16), dtype=torch.uint8, device=device)
    return {
        "crop_fwd/box_ind": lambda: ops.crop_and_resize_forward(maps[0], boxes, short, p, p),
        "crop_bwd/box_ind": lambda: ops.crop_and_resize_backward(grads, boxes, short, sizes[0]),
        "crop_bwd/grads_n": lambda: ops.crop_and_resize_backward(grads[:N - 1], boxes, ind, sizes[0]),
        "pyr_fwd/box_ind": lambda: ops.pyramid_crop_forward(maps, boxes, short, lvl, p, p),
        "pyr_fwd/level": lambda: ops.pyramid_crop_forward(maps, boxes, ind, lvl[:N - 1], p, p),
        "pyr_bwd/box_ind": lambda: ops.pyramid_crop_backward(grads, boxes, short, lvl, sizes),
        "pyr_bwd/level": lambda: ops.pyramid_crop_backward(grads, boxes, ind, lvl[:N - 1], sizes),
        "pyr_bwd/grads_n": lambda: ops.pyramid_crop_backward(grads[:N - 1], boxes, ind, lvl, sizes),
        "pyr_bwd/channels": lambda: ops.pyramid_crop_backward(grads, boxes, ind, lvl, [(B, C + 4, 16, 16), sizes[1]]),
        "pyr_bwd/batch": lambda: ops.pyramid_crop_backward(grads, boxes, ind, lvl, [sizes[0], (B + 1, C, 8, 8)]),
        "plan/box_ind": lambda: ops.pyramid_crop_backward_plan(boxes, short, lvl, sizes, C, p, p),
        "plan/level": lambda: ops.pyramid_crop_backward_plan(boxes, ind, lvl[:N - 1], sizes, C, p, p),
        "plan/channels": lambda: ops.pyramid_crop_backward_plan(boxes, ind, lvl, sizes, C + 4, p, p),
        "mask_targets/assignment": lambda: ops.mask_targets_device(masks, short, boxes, 28, 28),
    }


@gpu
def test_length_mismatches_raise_before_any_launch():
    from sln_amodal_b200 import _lib, ops
    for what, call in _mismatched_calls(ops, dev()).items():
        l0 = _lib.launches()
        with pytest.raises(_lib.SlnError):
            call()
        assert _lib.launches() == l0, what
    torch.cuda.synchronize()


# ---- the same contract without a GPU: CPU tensors, and a library stub that fails the test when anything reaches it
class _LibStub:
    def __init__(self, **allowed):
        self._allowed = allowed

    def __getattr__(self, name):
        if name in self._allowed:
            return self._allowed[name]

        def called(*args):
            raise AssertionError(f"{name} was called: the ops layer let the call through to the kernels")
        return called


@pytest.fixture
def cpu_ops(monkeypatch):
    from sln_amodal_b200 import ops
    monkeypatch.setattr(ops, "_require_cuda", lambda t, name: None)
    monkeypatch.setattr(ops, "lib", lambda: _LibStub())
    return ops


def test_length_mismatches_raise_without_gpu(cpu_ops):
    from sln_amodal_b200 import _lib
    missed = []
    for what, call in _mismatched_calls(cpu_ops, torch.device("cpu")).items():
        l0 = _lib.launches()
        try:
            call()
            missed.append(f"{what}: no error")
        except _lib.SlnError:
            if _lib.launches() != l0:
                missed.append(f"{what}: launches counted")
        except Exception as e:                   # reached the stub, or CUDA-only code further down
            missed.append(f"{what}: {type(e).__name__}")
    assert not missed, missed


@pytest.mark.parametrize("dtype", NON_F32, ids=_dtype_id)
def test_layout_converters_return_f32_without_gpu(cpu_ops, dtype):
    """to_channels_last / to_contiguous_nchw give f32 whatever the input dtype; these inputs need no transpose."""
    x = torch.randn(2, 5, 3, 4).to(dtype)
    cl = x.contiguous(memory_format=torch.channels_last)
    y = cpu_ops.to_channels_last(cl)
    assert y.dtype == torch.float32 and cpu_ops.is_channels_last(y) and torch.equal(y, x.float())
    y = cpu_ops.to_contiguous_nchw(x)
    assert y.dtype == torch.float32 and y.is_contiguous() and torch.equal(y, x.float())


@pytest.mark.parametrize("dtype", NON_F32, ids=_dtype_id)
def test_pyramid_forward_hands_f32_maps_to_the_kernel_without_gpu(cpu_ops, monkeypatch, dtype):
    """A channels_last map of another dtype reaches sln_pyramid_crop_fwd as an f32 NHWC copy of its values.  The stub
    reads the maps it is given (host memory here) before anything is launched."""
    seen = []

    def pyramid_fwd(mp, hs, ws, nl, B, C, *rest):
        for lv in range(nl):
            src = maps[lv]
            assert mp[lv] != src.data_ptr(), f"map {lv}: the {src.dtype} tensor itself was handed to the f32 kernel"
            n = B * C * hs[lv] * ws[lv]
            seen.append(np.ctypeslib.as_array((ctypes.c_float * n).from_address(mp[lv])).copy())
        return 0
    monkeypatch.setattr(cpu_ops, "lib", lambda: _LibStub(sln_pyramid_crop_fwd=pyramid_fwd))
    monkeypatch.setattr(cpu_ops, "stream_ptr", lambda: None)
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    maps = [torch.randn(2, 6, s, s + 1).to(dtype).contiguous(memory_format=torch.channels_last) for s in (5, 3)]
    boxes = torch.rand(4, 4)
    zeros = torch.zeros(4, dtype=torch.int32)
    cpu_ops.pyramid_crop_forward(maps, boxes, zeros, zeros, 7, 7)
    assert len(seen) == len(maps)
    for m, got in zip(maps, seen):
        assert got.tobytes() == m.float().permute(0, 2, 3, 1).contiguous().numpy().tobytes()
