"""unmold_detections_batched / ops.unmold_rle_batched_device against the single-image evaluation tail.

The single-image path -- unmold.unmold_detections(..., return_device_planes=True) followed by rle.encode(planes) -- is
pinned to Pillow and maskApi.c elsewhere (test_gpu_parity.py, test_oracle_pin.py).  Here every image's boxes, class ids
and scores must be bit-identical to it and every RLE string byte-identical.  The input-contract tests at the end run
without a device, against a stub of the library that fails when it is called.
"""
import contextlib
import ctypes as C

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu

MH = MW = 28
K = 3
# (image shape, window) pairs as the molding step produces them for a 1024^2 network input, plus odd ones
IMAGES = [((1024, 1024, 3), (0, 0, 1024, 1024)),
          ((480, 640, 3), (128, 0, 896, 1024)),
          ((1440, 1920, 3), (128, 0, 896, 1024)),
          ((130, 131, 3), (2, 0, 1022, 1024)),
          ((1024, 1024, 3), (0, 128, 1024, 896))]


def dev():
    return torch.device("cuda", 0)


def _blob(rng):
    yy, xx = np.mgrid[0:MH, 0:MW].astype(np.float32)
    cy, cx = rng.uniform(4, MH - 4, 2)
    s = rng.uniform(10, 80)
    return np.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / s).astype(np.float32) + 0.02 * rng.random((MH, MW), np.float32)


def _to_window(img_box, shape, window):
    """image-pixel box -> the network-input (molded) coordinates the detections carry"""
    sy = (window[2] - window[0]) / shape[0]
    sx = (window[3] - window[1]) / shape[1]
    y1, x1, y2, x2 = img_box
    return [y1 * sy + window[0], x1 * sx + window[1], y2 * sy + window[0], x2 * sx + window[1]]


def _make_batch(B, D, seed, specials=True):
    """B images (cycling through IMAGES) of D detection rows: special rows first (dropped boxes, whole image, 1 pixel,
    smaller than the mask, constant mask, two full-height neighbours, a noise mask), random blob detections, then the
    padding cut and rows behind it that must be ignored."""
    rng = np.random.default_rng(seed)
    det = np.zeros((B, D, 6), np.float32)
    mm = np.zeros((B, D, MH, MW, K), np.float32)
    shapes, windows = [], []
    for b in range(B):
        shape, window = IMAGES[b % len(IMAGES)]
        shapes.append(shape)
        windows.append(window)
        H, W = shape[:2]
        for d in range(D):
            for k in range(K):
                mm[b, d, :, :, k] = _blob(rng)
        rows = []
        if specials:
            rows += [
                ("zero area", _to_window((10, 10, 10, 40), shape, window)),
                ("inverted", _to_window((50, 40, 20, 60), shape, window)),
                ("past the border", _to_window((H - 5, 3, H + 3, 40), shape, window)),
                ("whole image", list(window)),
                ("one pixel", _to_window((H // 2, W // 3, H // 2 + 1, W // 3 + 1), shape, window)),
                ("small", _to_window((H // 4, W // 5, H // 4 + 17, W // 5 + 11), shape, window)),
                ("constant", _to_window((H // 3, W // 4, H // 3 + H // 3, W // 4 + W // 5), shape, window)),
                ("full height left", [window[0], _to_window((0, W // 4, H, W // 2), shape, window)[1], window[2],
                                      _to_window((0, W // 4, H, W // 2), shape, window)[3]]),
                ("full height right", [window[0], _to_window((0, W // 2, H, 3 * W // 4), shape, window)[1], window[2],
                                       _to_window((0, W // 2, H, 3 * W // 4), shape, window)[3]]),
                ("noise", _to_window((H // 10, W // 10, H // 10 + min(H, 400) * 8 // 10, W // 10 + min(W, 400) * 8 // 10),
                                     shape, window)),
            ]
        n = int(rng.integers(len(rows) + 5, D - 3)) if D > len(rows) + 8 else len(rows)
        for d in range(n):
            if d < len(rows):
                what, box = rows[d]
                det[b, d, :4] = box
                if what == "constant":
                    mm[b, d, :, :, 1] = 0.3
                elif what.startswith("full height"):
                    ramp = np.abs(np.arange(MH, dtype=np.float32) - (MH - 1) / 2) / ((MH - 1) / 2)
                    mm[b, d, :, :, 1] = ramp[:, None]            # ones at the top and bottom rows: runs merge across columns
                elif what == "noise":
                    mm[b, d, :, :, 1] = rng.random((MH, MW), np.float32)
            else:
                bh, bw = np.exp(rng.uniform(np.log(4), np.log(600), 2))
                y1 = rng.uniform(window[0], max(window[0] + 1, window[2] - bh))
                x1 = rng.uniform(window[1], max(window[1] + 1, window[3] - bw))
                det[b, d, :4] = [y1, x1, min(y1 + bh, window[2]), min(x1 + bw, window[3])]
            det[b, d, 4] = rng.integers(1, 6)
            det[b, d, 5] = rng.random()
        if n < D:                                            # padding cut at n; rows behind it look valid but are ignored
            det[b, n + 1:, :4] = det[b, : D - n - 1, :4]
            det[b, n + 1:, 4] = 2
            det[b, n + 1:, 5] = 0.5
    return det, mm, shapes, windows


def _single(det_b, mm_b, shape, window):
    from sln_amodal_b200 import rle, unmold
    boxes, cls, scores, planes = unmold.unmold_detections(det_b, mm_b, shape, np.asarray(window), return_device_planes=True)
    return boxes, cls, scores, (rle.encode(planes) if boxes.shape[0] else [])


def _assert_same(got, det, mm, shapes, windows):
    assert len(got) == det.shape[0]
    for b in range(det.shape[0]):
        want = _single(det[b], mm[b], shapes[b], windows[b])
        for g, w, name in zip(got[b][:3], want[:3], ("boxes", "class_ids", "scores")):
            assert g.dtype == w.dtype and g.shape == w.shape and np.array_equal(g, w), (b, name, g, w)
        assert len(got[b][3]) == len(want[3]), b
        for k, (g, w) in enumerate(zip(got[b][3], want[3])):
            assert g == w, (b, k, got[b][0][k].tolist())


@gpu
@pytest.mark.parametrize("B", [1, 3, 8])
def test_batched_matches_single_image(B):
    from sln_amodal_b200 import unmold_detections_batched
    det, mm, shapes, windows = _make_batch(B, 100, seed=B)
    T, M = torch.from_numpy(det).to(dev()), torch.from_numpy(mm).to(dev())
    got = unmold_detections_batched(T, M, shapes, windows)
    _assert_same(got, T, M, shapes, windows)
    # the special rows did what they are there for: drops, and at least one overflow retry in a 1024-wide image
    from sln_amodal_b200 import ops
    out = ops.unmold_rle_batched_device(T, M, shapes, windows)
    m = out.m.cpu().numpy()
    nk = out.num_kept.cpu().numpy()
    assert (m[0, : nk[0]] < 0).sum() >= 1 and (m[0, : nk[0]] > 0).sum() >= 10
    assert all(len(got[b][0]) <= 100 - 3 for b in range(B))


@gpu
def test_small_cap_retries_every_mask():
    """cap = 2: nearly every mask overflows and is re-encoded through unmold_masks + rle.encode; same results."""
    from sln_amodal_b200 import unmold_detections_batched
    det, mm, shapes, windows = _make_batch(2, 30, seed=7)
    T, M = torch.from_numpy(det).to(dev()), torch.from_numpy(mm).to(dev())
    _assert_same(unmold_detections_batched(T, M, shapes, windows, cap=2), T, M, shapes, windows)


@gpu
def test_permuted_mask_layout():
    """A permuted view of a head's [B, D, K, h, w] output is read through its strides, without a copy."""
    from sln_amodal_b200 import unmold_detections_batched
    det, mm, shapes, windows = _make_batch(3, 40, seed=11)
    T = torch.from_numpy(det).to(dev())
    head = torch.from_numpy(np.ascontiguousarray(mm.transpose(0, 1, 4, 2, 3))).to(dev())
    view = head.permute(0, 1, 3, 4, 2)
    assert not view.is_contiguous()
    got = unmold_detections_batched(T, view, shapes, windows)
    _assert_same(got, T, view.contiguous(), shapes, windows)


@gpu
def test_empty_images_and_empty_batch():
    from sln_amodal_b200 import ops, unmold_detections_batched
    det, mm, shapes, windows = _make_batch(3, 20, seed=5)
    det[1, :, 4] = 0                                          # image 1: the cut at row 0
    det[2, :, :4] = 0                                         # image 2: every box has zero area
    T, M = torch.from_numpy(det).to(dev()), torch.from_numpy(mm).to(dev())
    got = unmold_detections_batched(T, M, shapes, windows)
    for b in (1, 2):
        boxes, cls, scores, rles = got[b]
        want = _single(T[b], M[b], shapes[b], windows[b])
        assert boxes.shape == (0, 4) and boxes.dtype == np.int32 and cls.dtype == np.int32 and scores.dtype == np.float32
        assert np.array_equal(boxes, want[0]) and np.array_equal(cls, want[1]) and np.array_equal(scores, want[2])
        assert rles == []
    _assert_same(got[:1], T[:1], M[:1], shapes[:1], windows[:1])
    assert unmold_detections_batched(T[:0], M[:0], [], []) == []
    out = ops.unmold_rle_batched_device(T[:, :0], M[:, :0], shapes, windows)
    assert out.num_kept.cpu().tolist() == [0, 0, 0] and int(out.str_total.item()) == 0


_COUNT_KERNELS = """
import json, sys, numpy as np, torch
from torch.profiler import ProfilerActivity, profile
sys.path.insert(0, "tests")
from test_unmold_rle_batched import _make_batch
from sln_amodal_b200 import ops
counts = {}
for B in (1, 8):
    det, mm, shapes, windows = _make_batch(B, 100, seed=3)
    T, M = torch.from_numpy(det).cuda(), torch.from_numpy(mm).cuda()
    ops.unmold_rle_batched_device(T, M, shapes, windows)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ops.unmold_rle_batched_device(T, M, shapes, windows)
        torch.cuda.synchronize()
    c = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and "memset" not in e.name.lower() and "memcpy" not in e.name.lower():
            c[e.name] = c.get(e.name, 0) + 1
    counts[B] = c
print(json.dumps(counts))
"""


@gpu
def test_launches_do_not_depend_on_batch():
    """The same five kernels, once each, for B = 1 and B = 8 (torch.profiler in a fresh process: a long test process
    that has already run other profiler sessions can come back with no CUDA events)."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _COUNT_KERNELS], cwd=root, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    counts = json.loads(r.stdout.strip().splitlines()[-1])
    assert counts["1"] == counts["8"] and len(counts["1"]) == 5 and all(v == 1 for v in counts["1"].values()), counts


@gpu
def test_graph_capture_replays_the_eager_call():
    from sln_amodal_b200 import ops
    det, mm, shapes, windows = _make_batch(3, 100, seed=13)
    T, M = torch.from_numpy(det).to(dev()), torch.from_numpy(mm).to(dev())
    eager = ops.unmold_rle_batched_device(T, M, shapes, windows)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.unmold_rle_batched_device(T, M, shapes, windows)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        cap = ops.unmold_rle_batched_device(T, M, shapes, windows)
    cap.meta.fill_(-7)
    cap.strings.fill_(0)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(cap.meta, eager.meta)
    n = int(eager.str_total.item())
    assert n > 0 and torch.equal(cap.strings[:n], eager.strings[:n])


@gpu
def test_device_string_coder_matches_maskapi():
    """sln_rle_strings against oracle.rle_to_string: values near 2^32, negative deltas, short lists (the delta starts
    at index 3), an empty list and one with more runs than its capacity."""
    from oracle import oracle
    from sln_amodal_b200 import ops
    rng = np.random.default_rng(17)
    top = 2 ** 32 - 1
    lists = [[top, 0, top, 1, top - 5, 2, 0, top],
             [5], [0, 7], [3, 1, 4],
             [0, top, 0, top, 0, top, 1, 2],
             list(rng.integers(0, 2 ** 32, 500, dtype=np.uint64)),
             list(rng.integers(0, 40, 300)),
             [],
             [1, 2, 3]]
    cap = max(len(v) for v in lists)
    counts = np.zeros((len(lists), cap), np.uint32)
    m = np.zeros(len(lists), np.int32)
    for i, v in enumerate(lists):
        counts[i, : len(v)] = v
        m[i] = len(v)
    m[-1] = -3                                                # an overflowed mask: no string
    strings, off, slen, total = ops.rle_strings_device(torch.from_numpy(counts.view(np.int32)).to(dev()),
                                                       torch.from_numpy(m).to(dev()))
    s = strings.cpu().numpy().tobytes()
    off, slen = off.cpu().numpy(), slen.cpu().numpy()
    assert int(total.item()) == int(slen.sum())
    for i, v in enumerate(lists):
        want = oracle.rle_to_string(v) if m[i] > 0 else b""
        assert s[off[i]: off[i] + slen[i]] == want, i


# ---- input contract without a GPU: CPU tensors, and a library stub that fails the test when anything reaches it
class _LibStub:
    def __getattr__(self, name):
        def called(*args):
            raise AssertionError(f"{name} was called: the ops layer let the call through to the kernels")
        return called


@pytest.fixture
def cpu_ops(monkeypatch):
    from sln_amodal_b200 import ops
    monkeypatch.setattr(ops, "_require_cuda", lambda t, name: None)
    monkeypatch.setattr(ops, "lib", lambda: _LibStub())
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    return ops


def _bad_calls(ops):
    det, mm = torch.zeros(2, 10, 6), torch.zeros(2, 10, 28, 28, 3)
    shapes, windows = [(64, 64, 3)] * 2, [(0, 0, 64, 64)] * 2
    call = ops.unmold_rle_batched_device
    return {
        "2-D detections": lambda: call(det[0], mm, shapes, windows),
        "detections last dim": lambda: call(torch.zeros(2, 10, 5), mm, shapes, windows),
        "f64 detections": lambda: call(det.double(), mm, shapes, windows),
        "4-D masks": lambda: call(det, mm[0], shapes, windows),
        "f16 masks": lambda: call(det, mm.half(), shapes, windows),
        "masks B": lambda: call(det, torch.zeros(3, 10, 28, 28, 3), shapes, windows),
        "masks D": lambda: call(det, torch.zeros(2, 9, 28, 28, 3), shapes, windows),
        "image_shapes B": lambda: call(det, mm, shapes[:1], windows),
        "windows B": lambda: call(det, mm, shapes, windows * 2),
        "mask too large": lambda: call(det, torch.zeros(2, 10, 300, 28, 3), shapes, windows),
        "image side 0": lambda: call(det, mm, [(0, 64, 3), (64, 64, 3)], windows),
        "float32 window": lambda: call(det, mm, shapes, [np.array([0, 0, 64, 64], np.float32)] * 2),
        "cap 0": lambda: call(det, mm, shapes, windows, cap=0),
        "B over the limit": lambda: call(torch.zeros(513, 1, 6), torch.zeros(513, 1, 28, 28, 3), [(64, 64)] * 513,
                                         [(0, 0, 64, 64)] * 513),
        "coder counts 1-D": lambda: ops.rle_strings_device(torch.zeros(5, dtype=torch.int32), torch.zeros(5, dtype=torch.int32)),
        "coder m length": lambda: ops.rle_strings_device(torch.zeros(5, 4, dtype=torch.int32), torch.zeros(4, dtype=torch.int32)),
    }


def test_unmold_rle_batched_contract_raises_without_gpu(cpu_ops):
    from sln_amodal_b200 import _lib
    missed = []
    for what, call in _bad_calls(cpu_ops).items():
        l0 = _lib.launches()
        try:
            call()
            missed.append(f"{what}: no error")
        except _lib.SlnError:
            if _lib.launches() != l0:
                missed.append(f"{what}: launches counted")
        except Exception as e:                   # reached the stub, or CUDA-only code further down
            missed.append(f"{what}: {type(e).__name__}: {e}")
    assert not missed, missed


def test_scale_shift_is_the_references_arithmetic():
    from sln_amodal_b200 import ops
    for shape, window in IMAGES:
        h = shape[0] / (window[2] - window[0])
        w = shape[1] / (window[3] - window[1])
        assert ops.unmold_scale_shift(shape, window) == (h, w, float(window[0]), float(window[1]))
        assert ops.unmold_scale_shift(shape, np.asarray(window, np.int32)) == (h, w, float(window[0]), float(window[1]))


@pytest.fixture(scope="module")
def built_lib():
    from sln_amodal_b200 import build
    return build.build()


def test_new_symbols_reject_bad_arguments(built_lib):
    """Argument checks of the two new entry points run before any CUDA call and leave an error string."""
    from sln_amodal_b200 import _lib
    L = _lib.lib()
    H = (C.c_int * 2)(64, 64)
    W = (C.c_int * 2)(64, 0)
    assert L.sln_unmold_rle_batched_workspace_bytes(2, 10, H, (C.c_int * 2)(64, 64), 129) >= 2 * 10 * 64 * 64
    assert L.sln_unmold_rle_batched_workspace_bytes(2, 10, H, W, 129) == 0
    st = (C.c_longlong * 5)(0, 0, 0, 0, 0)
    sa = (C.c_double * 8)(*([1.0] * 8))
    args = lambda B, mh, Wa, cap, scap: (None, B, 10, None, mh, 28, 3, st, H, Wa, sa, cap) + (None,) * 10 + \
        (scap, None, 0, None)
    rc = L.sln_unmold_rle_batched(*args(2, 28, (C.c_int * 2)(64, 64), 0, 1 << 20))
    assert rc == -1 and b"cap" in L.sln_last_error_string()
    rc = L.sln_unmold_rle_batched(*args(2, 400, (C.c_int * 2)(64, 64), 129, 1 << 20))
    assert rc == -1 and b"mask" in L.sln_last_error_string()
    rc = L.sln_unmold_rle_batched(*args(2, 28, W, 129, 1 << 20))
    assert rc == -1 and b"image 1" in L.sln_last_error_string()
    rc = L.sln_unmold_rle_batched(*args(2, 28, (C.c_int * 2)(64, 64), 129, 100))
    assert rc == -1 and b"strings_cap" in L.sln_last_error_string()
    rc = L.sln_unmold_rle_batched(*args(600, 28, (C.c_int * 2)(64, 64), 129, 1 << 20))
    assert rc == -1 and b"512" in L.sln_last_error_string()
    rc = L.sln_rle_strings(None, 4, 0, None, None, None, None, None, 1 << 20, None)
    assert rc == -1 and b"cap" in L.sln_last_error_string()
    rc = L.sln_rle_strings(None, 4, 8, None, None, None, None, None, 10, None)
    assert rc == -1 and b"strings_cap" in L.sln_last_error_string()
