"""The batched NMS (sln_nms_batched), refine_detections_batched and the graph heads' per-class NMS branch against
their single-image forms.

The single-image entry points are pinned to the oracle and the golden files elsewhere (test_gpu_parity.py); here every
batched result is compared with them bit for bit (torch.equal), problem by problem.  The input-contract tests at the end
run without a device, against a stub of the library that fails when it is called.
"""
import contextlib

import numpy as np
import pytest
import torch

from sln_amodal_b200 import synth

gpu = pytest.mark.gpu

STD = (0.1, 0.1, 0.2, 0.2)
WINDOW = (0.0, 0.0, 1024.0, 1024.0)


def dev():
    return torch.device("cuda", 0)


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev())


def _problems(B, n, K, seed, ties=False):
    """B problems of n boxes: RPN-like boxes (whole-pixel coordinates when class-aware, like the refine step's rounded
    detections), scores a permutation of linspace or quantised to 256 levels, class ids in [0, K) or None."""
    rng = np.random.default_rng(seed)
    dets, cls = [], []
    for b in range(B):
        boxes = synth.nms_boxes(n, seed=seed + 7 * b, kind="rpn", rounded=K is not None)
        dets.append(np.concatenate([boxes, synth.nms_scores(n, seed=seed + 7 * b + 1, ties=ties)[:, None]], 1))
        if K is not None:
            cls.append(rng.integers(0, K, n).astype(np.int32))
    return np.stack(dets).astype(np.float32), (np.stack(cls) if K is not None else None)


def _assert_equals_per_problem(dets, cls, thresh, max_keep=0, dense_only=False):
    """nms_batched_device against nms_device on every problem alone; returns the path report."""
    from sln_amodal_b200 import ops
    D = cuda(dets)
    C = cuda(cls) if cls is not None else None
    keep, num, path = ops.nms_batched_device(D, thresh, class_ids=C, max_keep=max_keep, dense_only=dense_only,
                                             return_path=True)
    B, n = dets.shape[:2]
    mk = n if max_keep == 0 or max_keep > n else max_keep
    assert keep.shape == (B, mk) and keep.dtype == torch.int64 and num.shape == (B,) and path.shape == (B,)
    for b in range(B):
        wk, wn, wp = ops.nms_device(D[b], thresh, class_ids=None if C is None else C[b], max_keep=max_keep,
                                    dense_only=dense_only, return_path=True)
        k = int(wn.item())
        assert int(num[b]) == k, (b, int(num[b]), k)
        assert torch.equal(keep[b, :k], wk[:k]), b
        assert int(path[b]) == int(wp.item()), b
    return path.cpu().numpy()


@gpu
@pytest.mark.parametrize("K", [None, 81, 2], ids=["agnostic", "K81", "K2"])
@pytest.mark.parametrize("n", [40, 1000, 6000, 20000])
@pytest.mark.parametrize("B", [1, 3, 16])
def test_batched_nms_equals_per_image_nms(B, n, K):
    """Below the sparse minimum (n = 40), on the sparse path (1000, 6000) and at 20000, where the sparse path still runs
    and the dense fallback would take its two stages; thresholds 0.3 / 0.7, max_keep 0 (all) and 100."""
    dets, cls = _problems(B, n, K, seed=1000 + n + B)
    for thresh in (0.3, 0.7):
        for max_keep in (0, 100):
            path = _assert_equals_per_problem(dets, cls, thresh, max_keep)
            assert n >= 65 or not path.any(), path


@gpu
@pytest.mark.parametrize("K", [None, 81], ids=["agnostic", "K81"])
@pytest.mark.parametrize("B", [1, 3])
def test_batched_nms_dense_only_two_stage(B, K):
    """dense_only at n = 20000: every problem runs the two-stage dense pipeline with its own stage scratch."""
    dets, cls = _problems(B, 20000, K, seed=77 + B)
    for thresh, max_keep in ((0.7, 0), (0.3, 100)):
        assert not _assert_equals_per_problem(dets, cls, thresh, max_keep, dense_only=True).any()


@gpu
@pytest.mark.parametrize("K", [None, 81], ids=["agnostic", "K81"])
def test_batched_nms_tie_heavy_scores(K):
    """Scores quantised to 256 levels (the config-3 variant): ties are broken by the lower index in every problem."""
    dets, cls = _problems(5, 6000, K, seed=31, ties=True)
    for thresh in (0.3, 0.7):
        _assert_equals_per_problem(dets, cls, thresh)
        _assert_equals_per_problem(dets, cls, thresh, max_keep=100, dense_only=True)


@gpu
@pytest.mark.parametrize("K", [None, 81], ids=["agnostic", "K81"])
def test_batched_nms_mixed_sparse_and_dense_problems(K):
    """Problem 1 is near-copies of one box (more overlapping pairs than the sparse NMS budgets for) and problem 3 holds
    a NaN box: both leave the sparse pass, their neighbours stay on it, and every problem equals its single-image result,
    with dense_only too."""
    n = 5000
    dets, cls = _problems(5, n, K, seed=52)
    rng = np.random.default_rng(53)
    dets[1, :, :4] = (np.array([100, 100, 300, 300], np.float32) + rng.normal(0, 1.0, (n, 4))).astype(np.float32)
    if K is not None:
        cls[1] = 7                                               # one class: the copies really do overlap each other
    dets[3, 17, 0] = np.nan
    path = _assert_equals_per_problem(dets, cls, 0.7)
    assert list(path) == [1, 0, 1, 0, 1], path
    assert not _assert_equals_per_problem(dets, cls, 0.7, dense_only=True).any()
    _assert_equals_per_problem(dets, cls, 0.3, max_keep=100)


@gpu
def test_batched_nms_empty_shapes():
    from sln_amodal_b200 import ops
    keep, num = ops.nms_batched_device(torch.zeros((0, 100, 5), device=dev()), 0.7)
    assert keep.shape == (0, 100) and num.shape == (0,)
    keep, num, path = ops.nms_batched_device(torch.zeros((3, 0, 5), device=dev()), 0.7, return_path=True)
    assert keep.shape == (3, 0) and num.tolist() == [0, 0, 0] and path.tolist() == [0, 0, 0]


# --------------------------------------------------------------------------- refine_detections, USE_NMS = True
class _Cfg:
    RPN_BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
    IMAGE_SHAPE = np.array([1024, 1024, 3])
    USE_NMS = True
    DETECTION_MIN_CONFIDENCE = 0.0
    DETECTION_NMS_THRESHOLD = 0.3


def _cfg(use_nms=True, min_conf=0.0):
    c = _Cfg()
    c.USE_NMS, c.DETECTION_MIN_CONFIDENCE = use_nms, min_conf
    return c


def _refine_inputs(B, N, K, seed):
    """Image 1 (when B > 1) is all background; image 2 (when B > 2) has foreground scores below 0.3 only."""
    rng = np.random.default_rng(seed)
    rois = np.stack([synth.roi_boxes(N, seed=seed + b) for b in range(B)]).astype(np.float32)
    lg = rng.standard_normal((B, N, K)).astype(np.float32) * 3.0
    if B > 1:
        lg[1, :, 0] += 100.0
    e = np.exp(lg - lg.max(2, keepdims=True))
    probs = (e / e.sum(2, keepdims=True)).astype(np.float32)
    if B > 2:
        probs[2] = np.float32(1.0 / K)                             # every class ties: argmax 0 -> background...
        probs[2, : N // 2, 1] = np.float32(0.2)                    # ...except rows whose class 1 scores 0.2
        probs[2, : N // 2, 0] = np.float32(0.1)
    probs[0, :5] = probs[0, 0]                                     # exact ties across rows
    deltas = (rng.standard_normal((B, N, K, 4)) * 0.3).astype(np.float32)
    return rois, probs, deltas


def _assert_refine_equals_eager(rois, probs, deltas, cfg, D):
    from sln_amodal_b200 import refine_detections, refine_detections_batched
    R, P, Dl = cuda(rois), cuda(probs), cuda(deltas)
    det, keep, num = refine_detections_batched(R, P, Dl, WINDOW, cfg, max_detections=D)
    B = rois.shape[0]
    assert det.shape == (B, D, 6) and keep.shape == (B, D) and num.shape == (B,)
    for b in range(B):
        wd, wk = refine_detections(R[b], P[b], Dl[b], WINDOW, cfg)
        m = min(D, len(wk))
        assert int(num[b]) == m, (b, int(num[b]), len(wk))
        if m:
            assert torch.equal(det[b, :m], wd[:m]) and torch.equal(keep[b, :m], wk[:m]), b
        assert not det[b, m:].any() and not keep[b, m:].any(), b
    return det, keep, num


@gpu
@pytest.mark.parametrize("min_conf", [0.0, 0.3])
@pytest.mark.parametrize("K", [81, 61, 2])
def test_refine_detections_batched_per_class_nms_equals_eager(K, min_conf):
    """USE_NMS = True for four images: untruncated (D = N) and the first 100; one image all background, and with
    min_conf 0.3 one whose every foreground score is below it."""
    B, N = 4, 1000
    rois, probs, deltas = _refine_inputs(B, N, K, seed=K)
    cfg = _cfg(True, min_conf)
    det, _, num = _assert_refine_equals_eager(rois, probs, deltas, cfg, N)
    assert int(num[1]) == 0
    if min_conf:
        assert int(num[2]) == 0
    n0 = int(num[0])
    assert n0 > 1
    _assert_refine_equals_eager(rois, probs, deltas, cfg, 100 if n0 > 100 else n0 // 2)      # a prefix that truncates


@gpu
def test_refine_detections_batched_against_the_oracle():
    from oracle import oracle
    from sln_amodal_b200 import refine_detections_batched
    B, N, K = 2, 300, 81
    rois, probs, deltas = _refine_inputs(B, N, K, seed=5)
    det, keep, num = refine_detections_batched(cuda(rois), cuda(probs), cuda(deltas), WINDOW, _cfg(True, 0.0), max_detections=N)
    for b in range(B):
        wd, wk = oracle.refine_detections(rois[b], probs[b], deltas[b], WINDOW, min_confidence=0.0, nms_threshold=0.3)
        wd, wk = np.asarray(wd, np.float32), np.asarray(wk, np.int64)
        m = int(num[b])
        assert m == wk.size, b
        assert np.array_equal(keep[b, :m].cpu().numpy(), wk) and np.array_equal(det[b, :m].cpu().numpy(), wd.reshape(m, 6)), b


@gpu
def test_refine_detections_batched_without_nms_equals_topk():
    """USE_NMS = False: decode + refine_topk_batched_device, zero beyond the counts (DETECTION_MIN_CONFIDENCE ignored)."""
    from sln_amodal_b200 import ops, refine_detections_batched
    B, N, K, D = 3, 1000, 81, 100
    rois, probs, deltas = _refine_inputs(B, N, K, seed=9)
    R, P, Dl = cuda(rois), cuda(probs), cuda(deltas)
    det, keep, num = refine_detections_batched(R, P, Dl, WINDOW, _cfg(False, 0.7), max_detections=D)
    dets, _, class_ids, _ = ops.refine_decode_device(R.view(B * N, 4), P.view(B * N, K), Dl.view(B * N, K, 4), STD,
                                                     (1024, 1024), WINDOW, 0.0)
    wd, wk, wn = ops.refine_topk_batched_device(dets.view(B, N, 5), class_ids.view(B, N), D)
    assert torch.equal(num, wn)
    for b in range(B):
        m = int(wn[b])
        assert torch.equal(det[b, :m], wd[b, :m]) and torch.equal(keep[b, :m], wk[b, :m]), b
        assert not det[b, m:].any() and not keep[b, m:].any(), b


# --------------------------------------------------------------------------- graph heads with USE_NMS = True
class _GraphNmsCfg:
    IMAGE_SHAPE = np.array([1024, 1024, 3])
    RPN_BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
    BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
    RPN_NMS_THRESHOLD = 0.7
    POOL_SIZE = 7
    MASK_POOL_SIZE = 14
    USE_NMS = True
    DETECTION_MIN_CONFIDENCE = 0.0
    DETECTION_NMS_THRESHOLD = 0.3


def _graph_image(r, A, K, Cc, sides):
    fg = r.permutation(np.linspace(0, 1, A)).astype(np.float32)
    lg = r.standard_normal((1000, K)).astype(np.float32) * 3.0
    return {"probs": np.stack([1 - fg, fg], 1).astype(np.float32), "deltas": (r.standard_normal((A, 4)) * 0.5).astype(np.float32),
            "cls_probs": (np.exp(lg) / np.exp(lg).sum(1, keepdims=True)).astype(np.float32),
            "cls_deltas": (r.standard_normal((1000, K, 4)) * 0.3).astype(np.float32),
            "maps": [r.standard_normal((1, Cc, s_, s_), dtype=np.float32) for s_ in sides]}


@gpu
def test_head_graph_per_class_nms_equals_the_eager_drop_ins():
    """HeadGraph with USE_NMS = True against the drop-ins (proposal_layer -> pyramid_roi_align -> refine_detections ->
    pyramid_roi_align) over two replays with the inputs refreshed in place: the first max_detections detections, their
    keep indices and their mask-head crops are identical, zero beyond num_detections."""
    from sln_amodal_b200 import pipeline, proposal_layer, pyramid_roi_align, refine_detections
    A, K, Cc, D = 65472, 81, 64, 100
    cfg = _GraphNmsCfg()
    anchors = cuda(synth.nms_boxes(A, seed=4, kind="rpn"))
    sides = (128, 64, 32, 16)
    r = np.random.default_rng(17)
    img = _graph_image(r, A, K, Cc, sides)
    st = {k: cuda(v) for k, v in img.items() if k != "maps"}
    st["maps"] = [cuda(m).contiguous(memory_format=torch.channels_last) for m in img["maps"]]
    graph = pipeline.HeadGraph(anchors, cfg, st["maps"], st["probs"], st["deltas"], (st["cls_probs"], st["cls_deltas"]),
                               max_detections=D)
    for rep in range(2):
        if rep:
            img = _graph_image(r, A, K, Cc, sides)
            for k in ("probs", "deltas", "cls_probs", "cls_deltas"):
                st[k].copy_(cuda(img[k]))
            for m, src in zip(st["maps"], img["maps"]):
                m.copy_(cuda(src))
        out = graph.replay()
        torch.cuda.synchronize()
        k, nd = int(out["num_rois"].item()), int(out["num_detections"].item())
        rois = proposal_layer([st["probs"].unsqueeze(0).clone(), st["deltas"].unsqueeze(0).clone()], 1000, 0.7, anchors, cfg)
        assert rois.shape[1] == k and torch.equal(rois[0], out["rois"][:k])
        det, keep = refine_detections(rois[0], st["cls_probs"][:k], st["cls_deltas"][:k], WINDOW, cfg)
        assert nd == min(D, len(keep)) and nd > 0, rep
        assert torch.equal(det[:nd], out["detections"][:nd]) and not out["detections"][nd:].any(), rep
        assert torch.equal(keep[:nd], out["keep"][:nd]) and not out["keep"][nd:].any(), rep
        mask_in = pyramid_roi_align([(det[:nd, :4] / 1024.0).unsqueeze(0)] + st["maps"], 14, cfg.IMAGE_SHAPE)
        assert torch.equal(mask_in, out["mask_pooled"][:nd]), rep


@gpu
def test_batched_head_graph_per_class_nms_equals_per_image_head_graphs():
    """BatchedHeadGraph with USE_NMS = True over three images against each image's own HeadGraph, two replays with the
    inputs refreshed in place: every output below the counts is identical, zero beyond them."""
    from sln_amodal_b200 import pipeline
    A, K, Cc, B = 65472, 81, 64, 3
    cfg = _GraphNmsCfg()
    anchors = cuda(synth.nms_boxes(A, seed=4, kind="rpn"))
    sides = (128, 64, 32, 16)
    r = np.random.default_rng(43)
    imgs = [_graph_image(r, A, K, Cc, sides) for _ in range(B)]
    st = {k: cuda(np.stack([im[k] for im in imgs])) for k in ("probs", "deltas", "cls_probs", "cls_deltas")}
    st["maps"] = [cuda(np.concatenate([im["maps"][l] for im in imgs])).contiguous(memory_format=torch.channels_last)
                  for l in range(len(sides))]
    batched = pipeline.BatchedHeadGraph(anchors, cfg, st["maps"], st["probs"], st["deltas"], (st["cls_probs"], st["cls_deltas"]))
    one = {k: st[k][0].clone() for k in ("probs", "deltas", "cls_probs", "cls_deltas")}
    one["maps"] = [m[:1].clone().contiguous(memory_format=torch.channels_last) for m in st["maps"]]
    single = pipeline.HeadGraph(anchors, cfg, one["maps"], one["probs"], one["deltas"], (one["cls_probs"], one["cls_deltas"]))
    for rep in range(2):
        if rep:
            imgs = [_graph_image(r, A, K, Cc, sides) for _ in range(B)]
            for k in ("probs", "deltas", "cls_probs", "cls_deltas"):
                st[k].copy_(cuda(np.stack([im[k] for im in imgs])))
            for l, m in enumerate(st["maps"]):
                m.copy_(cuda(np.concatenate([im["maps"][l] for im in imgs])))
        out = batched.replay()
        torch.cuda.synchronize()
        for b in range(B):
            for k in ("probs", "deltas", "cls_probs", "cls_deltas"):
                one[k].copy_(st[k][b])
            for m, src in zip(one["maps"], st["maps"]):
                m.copy_(src[b:b + 1])
            w = single.replay()
            torch.cuda.synchronize()
            k, nd = int(w["num_rois"].item()), int(w["num_detections"].item())
            assert nd > 0 and int(out["num_rois"][b]) == k and int(out["num_detections"][b]) == nd, (rep, b)
            assert torch.equal(out["rois"][b], w["rois"]), (rep, b)
            assert torch.equal(out["pooled"][b, :k], w["pooled"][:k]), (rep, b)
            assert torch.equal(out["detections"][b], w["detections"]), (rep, b)
            assert torch.equal(out["keep"][b], w["keep"]), (rep, b)
            assert torch.equal(out["mask_pooled"][b, :nd], w["mask_pooled"][:nd]), (rep, b)
            assert not out["detections"][b, nd:].any() and not out["keep"][b, nd:].any(), (rep, b)


# --------------------------------------------------------------------------- launch counts
def _kernel_counts(fn):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    counts = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and "memset" not in e.name.lower() and "memcpy" not in e.name.lower():
            counts[e.name] = counts.get(e.name, 0) + 1
    return counts


@gpu
@pytest.mark.parametrize("K", [None, 81], ids=["agnostic", "K81"])
def test_batched_nms_launches_each_sparse_stage_once(K):
    """B = 1 and B = 8 launch rank, bin, pairs and resolve once each; only the guarded dense kernels (mask + scan at
    n = 1000) are launched once per problem."""
    from sln_amodal_b200 import ops
    c = {}
    for B in (1, 8):
        dets, cls = _problems(B, 1000, K, seed=300)
        D, C = cuda(dets), (cuda(cls) if cls is not None else None)
        c[B] = _kernel_counts(lambda: ops.nms_batched_device(D, 0.3, class_ids=C, max_keep=100))
    dense = {k for k in c[1] if "nms_mask_kernel" in k or "nms_scan_kernel" in k}
    assert len(dense) == 2, c[1]
    for k in dense:
        assert c[1][k] == 1 and c[8][k] == 8, (k, c[1][k], c[8].get(k))
    rest1 = {k: v for k, v in c[1].items() if k not in dense}
    rest8 = {k: v for k, v in c[8].items() if k not in dense}
    assert rest1 == rest8 and all(v == 1 for v in rest1.values()), (rest1, rest8)
    assert len(rest1) == 4, rest1                    # rank (with the gather), bin, pairs, resolve


# --------------------------------------------------------------------------- input contract without a GPU
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
    from sln_amodal_b200 import refine_detections_batched
    dets, cls = torch.rand(2, 10, 5), torch.ones(2, 10, dtype=torch.int32)
    keep, num = torch.zeros(2, 5, dtype=torch.int64), torch.zeros(2, dtype=torch.int32)
    rois, probs, deltas = torch.rand(2, 10, 4), torch.rand(2, 10, 3), torch.rand(2, 10, 3, 4)
    refine = lambda *x, **kw: refine_detections_batched(*x, WINDOW, _cfg(True), **kw)
    return {
        "nms 2-D dets": lambda: ops.nms_batched_device(dets[0], 0.5),
        "nms dets last dim": lambda: ops.nms_batched_device(torch.rand(2, 10, 4), 0.5),
        "nms integer dets": lambda: ops.nms_batched_device(dets.to(torch.int32), 0.5),
        "nms class_ids B": lambda: ops.nms_batched_device(dets, 0.5, class_ids=torch.ones(3, 10, dtype=torch.int32)),
        "nms class_ids n": lambda: ops.nms_batched_device(dets, 0.5, class_ids=torch.ones(2, 9, dtype=torch.int32)),
        "nms float class_ids": lambda: ops.nms_batched_device(dets, 0.5, class_ids=torch.ones(2, 10)),
        "nms negative max_keep": lambda: ops.nms_batched_device(dets, 0.5, max_keep=-1),
        "nms B too large": lambda: ops.nms_batched_device(torch.rand(65536, 1, 5), 0.5),
        "emit 2-D dets": lambda: ops.refine_nms_emit_batched_device(dets[0], cls, keep, num, 5),
        "emit class_ids": lambda: ops.refine_nms_emit_batched_device(dets, cls[:, :9], keep, num, 5),
        "emit keep B": lambda: ops.refine_nms_emit_batched_device(dets, cls, keep[:1], num, 5),
        "emit keep wider than N": lambda: ops.refine_nms_emit_batched_device(dets, cls, torch.zeros(2, 11, dtype=torch.int64), num, 5),
        "emit num B": lambda: ops.refine_nms_emit_batched_device(dets, cls, keep, num[:1], 5),
        "emit int32 keep": lambda: ops.refine_nms_emit_batched_device(dets, cls, keep.to(torch.int32), num, 5),
        "emit negative D": lambda: ops.refine_nms_emit_batched_device(dets, cls, keep, num, -1),
        "refine 2-D rois": lambda: refine(rois[0], probs, deltas),
        "refine probs B": lambda: refine(rois, probs[:1], deltas),
        "refine probs N": lambda: refine(rois, probs[:, :9], deltas),
        "refine deltas K": lambda: refine(rois, probs, torch.rand(2, 10, 4, 4)),
        "refine negative D": lambda: refine(rois, probs, deltas, max_detections=-1),
    }


def test_batched_nms_shape_mismatches_raise_without_gpu(cpu_ops):
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


def test_nms_batched_is_the_ops_function():
    import sln_amodal_b200
    from sln_amodal_b200 import ops
    assert sln_amodal_b200.nms_batched is ops.nms_batched_device

