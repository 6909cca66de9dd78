"""RoIAlign on bf16 / fp16 maps: the 2-byte kernels against the f32 kernels run on the widened maps and rounded.

Widening bf16 / fp16 to f32 is exact, and the 2-byte kernels run the f32 operation sequence on the widened values with
f32 accumulators and round each result once, so every case here is a BITWISE comparison with the f32 call `.to(D)`
(NaN payloads aside: NaN positions must agree).  Forward, exact backward and default backward; planned and unplanned.
The autocast tests check the rule of the autograd entry points: inside torch.autocast, bf16 / fp16 maps give crops and
gradients of their own dtype with today's values rounded; outside, nothing changes.
"""
import contextlib

import numpy as np
import pytest
import torch

from sln_amodal_b200 import synth

gpu = pytest.mark.gpu

LOWP = [torch.bfloat16, torch.float16]


def _id(d):
    return str(d).replace("torch.", "")


def dev():
    return torch.device("cuda", 0)


def cuda(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.to(dev())


def assert_bits(got, want, what=""):
    """Same dtype, shape and bits; NaN where the other has NaN (any payload)."""
    assert got.dtype == want.dtype and got.shape == want.shape, (what, got.dtype, want.dtype, got.shape, want.shape)
    g, w = got.detach().contiguous(), want.detach().contiguous()
    gn, wn = torch.isnan(g), torch.isnan(w)
    assert torch.equal(gn, wn), f"{what}: NaN positions differ"
    iv = torch.int16 if g.element_size() == 2 else torch.int32
    gb, wb = g.view(iv)[~gn], w.view(iv)[~wn]
    bad = int((gb != wb).sum())
    assert bad == 0, f"{what}: {bad} of {gb.numel()} elements differ"


def edge_boxes(N, seed):
    """ROIs partly outside the image, degenerate (y1 == y2), y-flipped and x-flipped."""
    boxes = synth.roi_boxes(N, seed=seed, outside_frac=0.2, degenerate_frac=0.1)
    boxes[::7] = boxes[::7][:, [2, 1, 0, 3]]
    boxes[::11] = boxes[::11][:, [0, 3, 2, 1]]
    return boxes


def lowp_values(shape, dtype, seed):
    """Random values of `dtype` that include +-0, bf16 / fp16 subnormals and (fp16) values next to the largest finite."""
    rng = np.random.default_rng(seed)
    v = rng.standard_normal(shape).astype(np.float32)
    flat = v.reshape(-1)
    k = flat.size
    idx = rng.permutation(k)
    flat[idx[: k // 50]] = 0.0
    flat[idx[k // 50: k // 25]] = -0.0
    tiny = 1e-39 if dtype == torch.bfloat16 else 3e-6           # subnormal in the dtype
    flat[idx[k // 25: k // 15]] = tiny * rng.standard_normal(k // 15 - k // 25)
    if dtype == torch.float16:
        flat[idx[k // 15: k // 10]] = 65504.0 * np.sign(rng.standard_normal(k // 10 - k // 15))
    return torch.from_numpy(v).to(dtype)


# --------------------------------------------------------------------------- forward
FWD_C = [3, 4, 6, 8, 64, 256, 260]
FWD_POOLS = [(7, 7), (14, 14), (1, 32), (33, 33)]


@gpu
@pytest.mark.parametrize("pool", FWD_POOLS, ids=lambda p: f"{p[0]}x{p[1]}")
@pytest.mark.parametrize("C", FWD_C)
@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
@pytest.mark.parametrize("dtype", LOWP, ids=_id)
def test_forward_matches_widened_f32(dtype, layout, C, pool):
    from sln_amodal_b200 import ops
    ph, pw = pool
    B, H, W = 3, 21, 26
    N = int(np.clip(400_000 // (C * ph * pw), 8, 96))
    fmt = torch.channels_last if layout == "channels_last" else torch.contiguous_format
    img = lowp_values((B, C, H, W), dtype, 5 + C).to(dev()).contiguous(memory_format=fmt)
    rng = np.random.default_rng(C + ph)
    boxes = cuda(edge_boxes(N, 3 + C))
    ind_np = rng.integers(0, B, N).astype(np.int32)
    ind_np[::9] = -1                                      # out-of-range rows: zeros
    ind_np[::13] = B
    ind = cuda(ind_np)
    got = ops.crop_and_resize_forward(img, boxes, ind, ph, pw, 1.5, keep_dtype=True)
    want = ops.crop_and_resize_forward(img.float(), boxes, ind, ph, pw, 1.5).to(dtype)
    assert_bits(got, want, "crop_and_resize_forward")

    maps = [lowp_values((B, C, s, s + 5), dtype, 40 + s).to(dev()).contiguous(memory_format=fmt) for s in (19, 9, 4, 1)]
    lv_np = rng.integers(0, 4, N).astype(np.int32)
    lv_np[::10] = 4                                       # out-of-range level: zeros
    lv_np[::17] = -1
    lv = cuda(lv_np)
    got = ops.pyramid_crop_forward(maps, boxes, ind, lv, ph, pw, 1.5, keep_dtype=True)
    want = ops.pyramid_crop_forward([m.float() for m in maps], boxes, ind, lv, ph, pw, 1.5).to(dtype)
    assert_bits(got, want, "pyramid_crop_forward")


@gpu
def test_forward_extrapolation_overflows_fp16_like_the_cast():
    """An extrapolation value outside fp16's range becomes inf, as the cast of the f32 crop does; bf16 rounds it."""
    from sln_amodal_b200 import ops
    boxes = cuda(edge_boxes(64, 8))
    ind = torch.zeros(64, dtype=torch.int32, device=dev())
    for dtype in LOWP:
        img = lowp_values((1, 64, 12, 15), dtype, 2).to(dev()).contiguous(memory_format=torch.channels_last)
        got = ops.crop_and_resize_forward(img, boxes, ind, 7, 7, 70000.0, keep_dtype=True)
        assert_bits(got, ops.crop_and_resize_forward(img.float(), boxes, ind, 7, 7, 70000.0).to(dtype), _id(dtype))
        if dtype == torch.float16:
            assert torch.isinf(got).any()


# --------------------------------------------------------------------------- backward
# (C, H, W, ph, pw, misaligned): the bulk-async stage configurations of test_crop_edges.py at 2-byte channel classes
# (one chunk, partial / full; two and three chunks), then shapes the 2-byte kernel does not take (f32 kernels + rounding)
_BWD = {}
for _C in (8, 120, 256, 264, 512):
    for _ph, _pw in ((8, 8), (5, 13), (1, 32), (32, 1), (32, 32)):
        _BWD[f"tma-C{_C}-{_ph}x{_pw}"] = (_C, 37, 45, _ph, _pw, False)
_BWD["fallback-C12-7x7"] = (12, 30, 30, 7, 7, False)
_BWD["fallback-C64-33x33"] = (64, 40, 40, 33, 33, False)
_BWD["fallback-misaligned-C256-14x14"] = (256, 40, 40, 14, 14, True)


def _bwd_case(cid, dtype, seed=0):
    C, H, W, ph, pw, mis = _BWD[cid]
    B = 2
    N = int(np.clip(1_000_000 // (C * ph * pw), 12, 64))
    rng = np.random.default_rng(seed + C + ph)
    boxes = cuda(edge_boxes(N, seed + 1))
    ind = cuda(rng.integers(0, B, N).astype(np.int32))
    g = lowp_values((N, ph, pw, C), dtype, seed + 7)
    if mis:
        buf = torch.empty(g.numel() + 1, dtype=dtype, device=dev())
        nhwc = buf[1:].view(N, ph, pw, C)
        nhwc.copy_(g)
        gt = nhwc.permute(0, 3, 1, 2)
        assert gt.data_ptr() % 16 == 2
    else:
        gt = g.to(dev()).permute(0, 3, 1, 2)
    assert gt.is_contiguous(memory_format=torch.channels_last)
    return (B, C, H, W), boxes, ind, gt


@gpu
@pytest.mark.parametrize("cid", list(_BWD))
@pytest.mark.parametrize("dtype", LOWP, ids=_id)
def test_backward_matches_widened_f32(dtype, cid):
    from sln_amodal_b200 import ops
    size, boxes, ind, g = _bwd_case(cid, dtype)
    for exact in (True, False):
        for cl in (True, False):
            got = ops.crop_and_resize_backward(g, boxes, ind, size, channels_last_out=cl, exact=exact, out_dtype=dtype)
            want = ops.crop_and_resize_backward(g.float(), boxes, ind, size, channels_last_out=cl, exact=exact).to(dtype)
            assert_bits(got, want, f"exact={exact} channels_last={cl}")
            assert ops.is_channels_last(got) == cl or got.shape[2] * got.shape[3] == 1


PYR_SIDES = [(700, 300), (256, 256), (64, 57), (1, 57), (57, 1), (1, 1), (9, 9), (3, 300)]


@gpu
@pytest.mark.parametrize("pool", [7, 14, 33])
@pytest.mark.parametrize("dtype", LOWP, ids=_id)
def test_pyramid_backward_eight_levels_planned_and_unplanned(dtype, pool):
    """Eight levels, level 5 without ROIs, out-of-range level / box_ind rows; exact and default; plan built by an f32
    PLAN_ONLY call serves the 2-byte call (a plan does not depend on the dtype)."""
    from sln_amodal_b200 import ops
    B, C, N = 2, 64, 300
    rng = np.random.default_rng(pool)
    boxes = cuda(edge_boxes(N, 21))
    ind_np = rng.integers(0, B, N).astype(np.int32)
    ind_np[::23] = B
    lv_np = rng.choice([0, 1, 2, 3, 4, 6, 7], N).astype(np.int32)
    lv_np[::19] = 8
    lv_np[::29] = -1
    ind, lv = cuda(ind_np), cuda(lv_np)
    sizes = [(B, C, h, w) for h, w in PYR_SIDES]
    g = lowp_values((N, pool, pool, C), dtype, pool).to(dev()).permute(0, 3, 1, 2)
    plan = ops.pyramid_crop_backward_plan(boxes, ind, lv, sizes, C, pool, pool)
    for exact in (True, False):
        want = [o.to(dtype) for o in ops.pyramid_crop_backward(g.float(), boxes, ind, lv, sizes, exact=exact)]
        for p in (None, plan):
            got = ops.pyramid_crop_backward(g, boxes, ind, lv, sizes, exact=exact, plan=p, out_dtype=dtype)
            for l, (a, b) in enumerate(zip(got, want)):
                assert_bits(a, b, f"level {l} exact={exact} planned={p is not None}")
    maps = [lowp_values(sz, dtype, 3 + k).to(dev()).contiguous(memory_format=torch.channels_last) for k, sz in enumerate(sizes)]
    got = ops.pyramid_crop_forward(maps, boxes, ind, lv, pool, pool, keep_dtype=True)
    assert_bits(got, ops.pyramid_crop_forward([m.float() for m in maps], boxes, ind, lv, pool, pool).to(dtype), "forward")


# --------------------------------------------------------------------------- kernel names
@gpu
@pytest.mark.parametrize("dtype", LOWP, ids=_id)
def test_native_shapes_run_the_2byte_kernels(dtype):
    """Channels_last 2-byte maps and grads at C % 8 == 0 run the 2-byte instantiations only: no f32 crop kernel and no
    dtype conversion on the device."""
    from torch.profiler import ProfilerActivity, profile
    from sln_amodal_b200 import ops
    tname = "__nv_bfloat16" if dtype == torch.bfloat16 else "__half"
    B, C, N = 2, 256, 200
    maps = [lowp_values((B, C, s, s), dtype, s).to(dev()).contiguous(memory_format=torch.channels_last) for s in (64, 32)]
    sizes = [tuple(m.shape) for m in maps]
    boxes = cuda(edge_boxes(N, 2))
    ind = torch.zeros(N, dtype=torch.int32, device=dev())
    lv = cuda(np.random.default_rng(0).integers(0, 2, N).astype(np.int32))
    grads = {p: lowp_values((N, C, p, p), dtype, p).to(dev()).contiguous(memory_format=torch.channels_last) for p in (7, 14)}
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for p in (7, 14):
            plan = ops.pyramid_crop_backward_plan(boxes, ind, lv, sizes, C, p, p)
            ops.pyramid_crop_forward(maps, boxes, ind, lv, p, p, keep_dtype=True)
            ops.pyramid_crop_backward(grads[p], boxes, ind, lv, sizes, plan=plan, out_dtype=dtype)
            ops.crop_and_resize_forward(maps[0], boxes, ind, p, p, keep_dtype=True)
            ops.crop_and_resize_backward(grads[p], boxes, ind, sizes[0], out_dtype=dtype)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    crop = [n for n in names if "crop_fwd" in n or "crop_bwd_tma" in n]
    assert any(f"crop_fwd_nhwc_kernel<{tname}, 8," in n for n in crop), crop
    assert any(f"crop_bwd_tma_b16_kernel<{tname}," in n for n in crop), crop
    assert all(tname in n for n in crop), [n for n in crop if tname not in n]
    assert not [n for n in names if "copy" in n.lower() or "elementwise" in n.lower()], names


# --------------------------------------------------------------------------- autocast through the autograd entry points
def _entry_points(dtype, seed=0):
    """name -> fn(maps) returning crops; maps: 4 maps [1, C, s, s] (single-map entry points use the first)."""
    from sln_amodal_b200 import pyramid_roi_align
    from sln_amodal_b200.crop_and_resize import CropAndResize, CropAndResizeFunction, RoIAlign
    from sln_amodal_b200.pyramid import pyramid_roi_align_batched, pyramid_roi_align_image
    N, pool = 120, 7
    boxes = cuda(synth.roi_boxes(N, seed=seed + 1, outside_frac=0.1))
    ind = torch.zeros(N, dtype=torch.int32, device=dev())
    px = boxes[:, [1, 0, 3, 2]] * 40.0                  # (x1, y1, x2, y2) in pixels of a 41 x 41 map
    return {
        "CropAndResizeFunction": lambda ms: CropAndResizeFunction(pool, pool, 0)(ms[0], boxes, ind),
        "CropAndResize": lambda ms: CropAndResize(pool, pool, 0)(ms[0], boxes, ind),
        "RoIAlign": lambda ms: RoIAlign(pool, pool, 0)(ms[0], px, ind),
        "pyramid_roi_align": lambda ms: pyramid_roi_align([boxes.unsqueeze(0)] + ms, pool, (256, 256, 3)),
        "pyramid_roi_align_batched": lambda ms: pyramid_roi_align_batched(boxes, ind, ms, pool, (256, 256, 3)),
        "pyramid_roi_align_image": lambda ms: pyramid_roi_align_image([boxes.unsqueeze(0), ms[0]], pool, (256, 256, 3)),
    }


ENTRY_POINTS = ["CropAndResizeFunction", "CropAndResize", "RoIAlign", "pyramid_roi_align", "pyramid_roi_align_batched",
                "pyramid_roi_align_image"]


@gpu
@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
@pytest.mark.parametrize("name", ENTRY_POINTS)
@pytest.mark.parametrize("dtype", LOWP, ids=_id)
def test_autocast_entry_points(dtype, name, layout):
    fmt = torch.channels_last if layout == "channels_last" else torch.contiguous_format
    C = 64
    base = [lowp_values((1, C, s, s), dtype, s).to(dev()).contiguous(memory_format=fmt) for s in (41, 21, 11, 6)]
    fn = _entry_points(dtype)[name]

    def run(autocast):
        ms = [m.detach().clone(memory_format=torch.preserve_format).requires_grad_(True) for m in base]
        ctx = torch.autocast(device_type="cuda", dtype=dtype) if autocast else contextlib.nullcontext()
        with ctx:
            out = fn(ms)
        w = lowp_values(tuple(out.shape), dtype, 99).to(dev())      # an upstream gradient the dtype represents exactly
        out.backward(w.to(out.dtype))
        return out.detach(), [m.grad for m in ms]

    out_ac, grads_ac = run(True)
    out_32, grads_32 = run(False)
    assert out_32.dtype == torch.float32                             # outside autocast: unchanged
    assert out_ac.dtype == dtype
    assert_bits(out_ac, out_32.to(dtype), "crops")
    for k, (a, b) in enumerate(zip(grads_ac, grads_32)):
        if b is None:
            assert a is None
            continue
        assert a.dtype == dtype and b.dtype == dtype
        assert_bits(a, b, f"grad of map {k}")


@gpu
def test_autocast_leaves_f32_and_mixed_maps_alone():
    from sln_amodal_b200 import pyramid_roi_align
    boxes = cuda(synth.roi_boxes(50, seed=3)).unsqueeze(0)
    ms32 = [torch.randn(1, 16, s, s, device=dev()) for s in (32, 16, 8, 4)]
    mixed = [ms32[0].bfloat16(), ms32[1], ms32[2].half(), ms32[3]]
    with torch.autocast(device_type="cuda", dtype=torch.bfloat16):
        a = pyramid_roi_align([boxes] + ms32, 7, (256, 256, 3))
        b = pyramid_roi_align([boxes] + mixed, 7, (256, 256, 3))
    assert a.dtype == torch.float32 and b.dtype == torch.float32
    assert torch.equal(b, pyramid_roi_align([boxes] + [m.float() for m in mixed], 7, (256, 256, 3)))


# --------------------------------------------------------------------------- full size
@gpu
@pytest.mark.parametrize("dtype", LOWP, ids=_id)
def test_config2_size_matches_widened_f32(dtype):
    """C = 256, P2-P5 (256^2 .. 32^2), 8 x 1000 ROIs, 7x7 and 14x14, backward planned: bitwise."""
    from sln_amodal_b200 import ops
    B, C, per = 8, 256, 1000
    boxes_np = synth.roi_boxes(B * per, seed=4321)
    lv = cuda((synth.fpn_level(boxes_np) - 2).astype(np.int32))
    boxes = cuda(boxes_np)
    ind = cuda(np.repeat(np.arange(B, dtype=np.int32), per))
    gen = torch.Generator(device=dev())
    gen.manual_seed(7)
    maps = [torch.randn((B, C, s, s), device=dev(), generator=gen).to(dtype).contiguous(memory_format=torch.channels_last)
            for s in (256, 128, 64, 32)]
    sizes = [tuple(m.shape) for m in maps]
    for p in (7, 14):
        plan = ops.pyramid_crop_backward_plan(boxes, ind, lv, sizes, C, p, p)
        got = ops.pyramid_crop_forward(maps, boxes, ind, lv, p, p, keep_dtype=True)
        assert_bits(got, ops.pyramid_crop_forward([m.float() for m in maps], boxes, ind, lv, p, p).to(dtype), f"fwd {p}")
        del got
        g = torch.randn((B * per, C, p, p), device=dev(), generator=gen).to(dtype).contiguous(memory_format=torch.channels_last)
        got = ops.pyramid_crop_backward(g, boxes, ind, lv, sizes, plan=plan, out_dtype=dtype)
        want = ops.pyramid_crop_backward(g.float(), boxes, ind, lv, sizes, plan=plan)
        for l, (a, b) in enumerate(zip(got, want)):
            assert_bits(a, b.to(dtype), f"bwd {p} level {l}")


# --------------------------------------------------------------------------- without a GPU: a library stub
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
    monkeypatch.setattr(ops, "stream_ptr", lambda: None)
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    return ops


@pytest.mark.parametrize("dtype", LOWP, ids=_id)
def test_lowp_length_mismatches_raise_without_gpu(cpu_ops, dtype):
    from sln_amodal_b200 import _lib
    B, C, N, p = 2, 8, 10, 7
    boxes = torch.rand((N, 4))
    ind = torch.zeros(N, dtype=torch.int32)
    lvl = torch.zeros(N, dtype=torch.int32)
    short = ind[:N - 1]
    maps = [torch.zeros((B, C, s, s), dtype=dtype).contiguous(memory_format=torch.channels_last) for s in (16, 8)]
    sizes = [tuple(m.shape) for m in maps]
    grads = torch.zeros((N, C, p, p), dtype=dtype).contiguous(memory_format=torch.channels_last)
    calls = {
        "crop_fwd/box_ind": lambda: cpu_ops.crop_and_resize_forward(maps[0], boxes, short, p, p, keep_dtype=True),
        "crop_bwd/box_ind": lambda: cpu_ops.crop_and_resize_backward(grads, boxes, short, sizes[0], out_dtype=dtype),
        "crop_bwd/grads_n": lambda: cpu_ops.crop_and_resize_backward(grads[:N - 1], boxes, ind, sizes[0], out_dtype=dtype),
        "pyr_fwd/box_ind": lambda: cpu_ops.pyramid_crop_forward(maps, boxes, short, lvl, p, p, keep_dtype=True),
        "pyr_fwd/level": lambda: cpu_ops.pyramid_crop_forward(maps, boxes, ind, lvl[:N - 1], p, p, keep_dtype=True),
        "pyr_bwd/box_ind": lambda: cpu_ops.pyramid_crop_backward(grads, boxes, short, lvl, sizes, out_dtype=dtype),
        "pyr_bwd/level": lambda: cpu_ops.pyramid_crop_backward(grads, boxes, ind, lvl[:N - 1], sizes, out_dtype=dtype),
        "pyr_bwd/grads_n": lambda: cpu_ops.pyramid_crop_backward(grads[:N - 1], boxes, ind, lvl, sizes, out_dtype=dtype),
        "pyr_bwd/channels": lambda: cpu_ops.pyramid_crop_backward(grads, boxes, ind, lvl, [(B, C + 8, 16, 16), sizes[1]],
                                                                  out_dtype=dtype),
    }
    missed = []
    for what, call in calls.items():
        l0 = _lib.launches()
        try:
            call()
            missed.append(f"{what}: no error")
        except _lib.SlnError:
            if _lib.launches() != l0:
                missed.append(f"{what}: launches counted")
        except Exception as e:
            missed.append(f"{what}: {type(e).__name__}: {e}")
    assert not missed, missed


@pytest.mark.parametrize("dtype", LOWP, ids=_id)
def test_keep_dtype_and_out_dtype_reach_the_ex_entry_points_without_gpu(cpu_ops, monkeypatch, dtype):
    """keep_dtype / out_dtype hand the 2-byte tensors themselves to the *_ex entry points with the dtype's code; the
    defaults still call the f32 entry points."""
    from sln_amodal_b200 import _lib
    code = {torch.bfloat16: _lib.DTYPE_BF16, torch.float16: _lib.DTYPE_F16}[dtype]
    B, C, N, p = 2, 16, 6, 7
    maps = [torch.randn(B, C, s, s + 1).to(dtype).contiguous(memory_format=torch.channels_last) for s in (5, 3)]
    sizes = [tuple(m.shape) for m in maps]
    boxes = torch.rand(N, 4)
    zeros = torch.zeros(N, dtype=torch.int32)
    grads = torch.randn(N, C, p, p).to(dtype).contiguous(memory_format=torch.channels_last)
    seen = []

    def rec(name, ret=0):
        def f(*args):
            seen.append((name, args))
            return ret
        return f
    stub = _LibStub(**{n: rec(n) for n in ("sln_crop_and_resize_fwd_ex", "sln_pyramid_crop_fwd_ex", "sln_crop_and_resize_bwd_ex",
                                           "sln_pyramid_crop_bwd_ex", "sln_crop_and_resize_fwd", "sln_pyramid_crop_fwd")},
                    sln_crop_and_resize_bwd_workspace_bytes=lambda *a: 64, sln_pyramid_crop_bwd_workspace_bytes=lambda *a: 64)
    monkeypatch.setattr(cpu_ops, "lib", lambda: stub)

    out = cpu_ops.crop_and_resize_forward(maps[0], boxes, zeros, p, p, keep_dtype=True)
    assert out.dtype == dtype
    name, args = seen.pop()
    assert name == "sln_crop_and_resize_fwd_ex" and args[0] == code and args[1].value == maps[0].data_ptr()
    out = cpu_ops.pyramid_crop_forward(maps, boxes, zeros, zeros, p, p, keep_dtype=True)
    assert out.dtype == dtype
    name, args = seen.pop()
    assert name == "sln_pyramid_crop_fwd_ex" and args[0] == code and args[1][0] == maps[0].data_ptr()
    gm = cpu_ops.crop_and_resize_backward(grads, boxes, zeros, sizes[0], out_dtype=dtype)
    assert gm.dtype == dtype
    name, args = seen.pop()
    assert name == "sln_crop_and_resize_bwd_ex" and args[0] == code and args[1].value == grads.data_ptr()
    gms = cpu_ops.pyramid_crop_backward(grads, boxes, zeros, zeros, sizes, out_dtype=dtype)
    assert all(g.dtype == dtype for g in gms)
    name, args = seen.pop()
    assert name == "sln_pyramid_crop_bwd_ex" and args[0] == code and args[1].value == grads.data_ptr()
    # defaults: the f32 entry points, f32 crops
    out = cpu_ops.crop_and_resize_forward(maps[0], boxes, zeros, p, p)
    assert out.dtype == torch.float32 and seen.pop()[0] == "sln_crop_and_resize_fwd"
    out = cpu_ops.pyramid_crop_forward(maps, boxes, zeros, zeros, p, p)
    assert out.dtype == torch.float32 and seen.pop()[0] == "sln_pyramid_crop_fwd"
    # mixed dtypes keep today's path even with keep_dtype
    out = cpu_ops.pyramid_crop_forward([maps[0], maps[1].float()], boxes, zeros, zeros, p, p, keep_dtype=True)
    assert out.dtype == torch.float32 and seen.pop()[0] == "sln_pyramid_crop_fwd"
