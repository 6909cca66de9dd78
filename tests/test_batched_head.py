"""The batched proposal layer, the batched detection top-k and BatchedHeadGraph against their single-image forms.

The single-image entry points are pinned to the oracle and the golden files elsewhere (test_gpu_parity.py,
test_golden.py); here every batched result is compared with them bit for bit (torch.equal), image by image.
The input-contract tests at the end run without a device, against a stub of the library that fails when it is called.
"""
import contextlib

import numpy as np
import pytest
import torch

from sln_amodal_b200 import synth

gpu = pytest.mark.gpu

STD = (0.1, 0.1, 0.2, 0.2)
HW = (1024, 1024)


def dev():
    return torch.device("cuda", 0)


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev())


# same generator as test_gpu_parity.py::_proposal_inputs
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


def _batch(A, B, seed, ties=False):
    """B images on one anchor set: each image its own scores and deltas."""
    _, _, anchors = _proposal_inputs(A, seed)
    probs, deltas = [], []
    for b in range(B):
        p, d, _ = _proposal_inputs(A, seed + 1 + b, ties)
        probs.append(p)
        deltas.append(d)
    return np.stack(probs), np.stack(deltas), anchors


def _assert_batched_equals_single(probs, deltas, anchors, count, thresh, pre_nms_limit=6000):
    from sln_amodal_b200 import ops
    P, D, An = cuda(probs), cuda(deltas), cuda(anchors)
    boxes, num = ops.proposal_batched_device(P, D, An, count, thresh, STD, HW, pre_nms_limit=pre_nms_limit)
    assert boxes.shape == (probs.shape[0], count, 4) and num.shape == (probs.shape[0],)
    for b in range(probs.shape[0]):
        want, wnum = ops.proposal_device(P[b], D[b], An, count, thresh, STD, HW, pre_nms_limit=pre_nms_limit)
        assert int(num[b]) == int(wnum[0]), b
        assert torch.equal(boxes[b], want), b          # every row: survivors and the zero padding
    return boxes, num


@gpu
@pytest.mark.parametrize("B", [1, 2, 5, 16])
def test_batched_proposals_equal_per_image_proposals(B):
    probs, deltas, anchors = _batch(261888, B, 100 + B)
    _assert_batched_equals_single(probs, deltas, anchors, 1000, 0.7)


@gpu
@pytest.mark.parametrize("A,count,ties", [(20000, 1000, True), (700, 1000, True), (5000, 6000, False)],
                         ids=["ties-A20000", "select_all-A700", "count-beyond-survivors"])
def test_batched_proposals_edge_shapes(A, count, ties):
    probs, deltas, anchors = _batch(A, 3, 200 + A % 97, ties)
    boxes, num = _assert_batched_equals_single(probs, deltas, anchors, count, 0.7)
    if count > min(A, 6000):
        assert (num < count).all()                     # more rows than candidates: the tail really is padding


@gpu
def test_batched_proposals_zero_count_and_empty_batch():
    from sln_amodal_b200 import ops
    probs, deltas, anchors = _batch(5000, 2, 7)
    boxes, num = ops.proposal_batched_device(cuda(probs), cuda(deltas), cuda(anchors), 0, 0.7, STD, HW)
    assert boxes.shape == (2, 0, 4) and not num.any()
    boxes, num = ops.proposal_batched_device(cuda(probs[:0]), cuda(deltas[:0]), cuda(anchors), 100, 0.7, STD, HW)
    assert boxes.shape == (0, 100, 4) and num.shape == (0,)


@gpu
def test_batched_proposals_mixed_sparse_and_dense_fallback():
    """One image of the batch leaves the sparse NMS (checked on its own candidates with nms_device(return_path=True)),
    its neighbours stay on it; every image still equals its single-image result.  The anchors are shared, so they come
    in two halves: ordinary anchors, and near-copies of one box (the `dup` case of
    test_nms_sparse_only_flag_and_host_retry: more overlapping pairs than the sparse NMS budgets for).  Image 2 scores
    the copies highest, the other images the ordinary half; pre_nms_limit is below either half."""
    from sln_amodal_b200 import ops
    A, H = 20000, 10000
    rng = np.random.default_rng(61)
    _, _, normal = _proposal_inputs(H, 60)
    dup = (np.array([100, 100, 300, 300], np.float32) + rng.normal(0, 1.0, (H, 4))).astype(np.float32)
    anchors = np.concatenate([normal, dup]).astype(np.float32)
    probs, deltas = [], []
    for b in range(4):
        fg = rng.permutation(np.linspace(0.0, 1.0, A)).astype(np.float32)
        top = np.arange(A) >= H if b == 2 else np.arange(A) < H
        fg = np.where(top, 0.5 + 0.5 * fg, 0.5 * fg).astype(np.float32)
        probs.append(np.stack([1 - fg, fg], 1))
        scale = 0.01 if b == 2 else 1.0
        deltas.append((rng.standard_normal((A, 4)) * scale).astype(np.float32))
    probs, deltas = np.stack(probs).astype(np.float32), np.stack(deltas)
    # the path each image's NMS takes, on its top-6000 decoded boxes in visiting order (a torch restatement of the
    # decode: close enough to decide the path, which depends on the overlap structure only)
    paths = []
    An = cuda(anchors)
    for b in range(4):
        p, d = cuda(probs[b]), cuda(deltas[b])
        order = torch.argsort(p[:, 1], descending=True, stable=True)[:6000]
        a, dl = An[order], d[order] * torch.tensor(STD, device=dev())
        h, w = a[:, 2] - a[:, 0], a[:, 3] - a[:, 1]
        cy, cx = a[:, 0] + 0.5 * h + dl[:, 0] * h, a[:, 1] + 0.5 * w + dl[:, 1] * w
        h, w = h * torch.exp(dl[:, 2]), w * torch.exp(dl[:, 3])
        bx = torch.stack([cy - 0.5 * h, cx - 0.5 * w, cy + 0.5 * h, cx + 0.5 * w], 1).clamp(0, 1024)
        score = torch.linspace(1, 0, 6000, device=dev())           # keeps the visiting order
        _, _, path = ops.nms_device(torch.cat([bx, score[:, None]], 1), 0.7, return_path=True)
        paths.append(int(path.item()))
    assert paths[2] == 0 and all(paths[b] == 1 for b in (0, 1, 3)), paths
    _assert_batched_equals_single(probs, deltas, anchors, 1000, 0.7)


@gpu
def test_batched_proposals_all_dense_below_sparse_threshold():
    probs, deltas, anchors = _batch(20000, 3, 81)
    _assert_batched_equals_single(probs, deltas, anchors, 1000, 0.03)


@gpu
def test_batched_topk_equals_per_image_topk():
    from sln_amodal_b200 import ops
    B, N, K, D = 4, 1000, 9, 100
    rng = np.random.default_rng(90)
    rois = cuda(np.sort(rng.uniform(0, 1, (B * N, 2, 2)), axis=1).reshape(B * N, 4).astype(np.float32))     # (y1,x1,y2,x2)
    lg = rng.standard_normal((B * N, K)).astype(np.float32) * 3.0
    lg[:N // 2, 0] += 50.0                           # image 0: half its rows background
    lg[2 * N:3 * N, 0] += 100.0                      # image 2: every row background
    e = np.exp(lg - lg.max(1, keepdims=True))
    probs = cuda((e / e.sum(1, keepdims=True)).astype(np.float32))
    probs[3 * N + 5] = probs[3 * N + 7]              # image 3: a score tie
    deltas = cuda((rng.standard_normal((B * N, K, 4)) * 0.3).astype(np.float32))
    dets, _, class_ids, _ = ops.refine_decode_device(rois, probs, deltas, STD, HW, (0.0, 0.0, 1024.0, 1024.0), 0.0)
    res, keep, num = ops.refine_topk_batched_device(dets.view(B, N, 5), class_ids.view(B, N), D)
    assert int(num[2]) == 0
    for b in range(B):
        d_b, c_b = dets[b * N:(b + 1) * N], class_ids[b * N:(b + 1) * N]
        want_n = min(D, int(((c_b > 0) & (d_b[:, 4] > -float("inf"))).sum()))
        w_res, w_keep = ops.refine_topk_device(d_b, c_b, D)
        n = int(num[b])
        assert n == want_n, b
        assert torch.equal(res[b, :n], w_res[:n]) and torch.equal(keep[b, :n], w_keep[:n]), b


class _GraphCfg:
    IMAGE_SHAPE = np.array([1024, 1024, 3])
    RPN_BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
    BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
    RPN_NMS_THRESHOLD = 0.7
    POOL_SIZE = 7
    MASK_POOL_SIZE = 14


def _graph_image(r, A, K, Cc, sides):
    fg = r.permutation(np.linspace(0, 1, A)).astype(np.float32)
    lg = r.standard_normal((1000, K)).astype(np.float32) * 3.0
    return {"probs": np.stack([1 - fg, fg], 1).astype(np.float32), "deltas": (r.standard_normal((A, 4)) * 0.5).astype(np.float32),
            "cls_probs": (np.exp(lg) / np.exp(lg).sum(1, keepdims=True)).astype(np.float32),
            "cls_deltas": (r.standard_normal((1000, K, 4)) * 0.3).astype(np.float32),
            "maps": [r.standard_normal((1, Cc, s_, s_), dtype=np.float32) for s_ in sides]}


@gpu
def test_batched_head_graph_equals_per_image_head_graphs():
    """BatchedHeadGraph over three images against each image's own HeadGraph, replayed twice with the inputs refreshed
    in place: every output below the counts is identical, rois and detections are zero beyond them."""
    from sln_amodal_b200 import pipeline
    A, K, Cc, B = 65472, 9, 64, 3
    cfg = _GraphCfg()
    anchors = cuda(synth.nms_boxes(A, seed=4, kind="rpn"))
    sides = (128, 64, 32, 16)
    r = np.random.default_rng(41)
    imgs = [_graph_image(r, A, K, Cc, sides) for _ in range(B)]
    st = {k: cuda(np.stack([im[k] for im in imgs])) for k in ("probs", "deltas", "cls_probs", "cls_deltas")}
    st["maps"] = [cuda(np.concatenate([im["maps"][l] for im in imgs])).contiguous(memory_format=torch.channels_last)
                  for l in range(len(sides))]
    batched = pipeline.BatchedHeadGraph(anchors, cfg, st["maps"], st["probs"], st["deltas"], (st["cls_probs"], st["cls_deltas"]))
    one = {"probs": cuda(imgs[0]["probs"]), "deltas": cuda(imgs[0]["deltas"]), "cls_probs": cuda(imgs[0]["cls_probs"]),
           "cls_deltas": cuda(imgs[0]["cls_deltas"]),
           "maps": [cuda(m).contiguous(memory_format=torch.channels_last) for m in imgs[0]["maps"]]}
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
            assert int(out["num_rois"][b]) == k and int(out["num_detections"][b]) == nd, (rep, b)
            assert torch.equal(out["rois"][b], w["rois"]), (rep, b)
            assert torch.equal(out["pooled"][b, :k], w["pooled"][:k]), (rep, b)
            assert torch.equal(out["detections"][b], w["detections"]), (rep, b)
            assert torch.equal(out["keep"][b, :nd], w["keep"][:nd]) and not out["keep"][b, nd:].any(), (rep, b)
            assert torch.equal(out["mask_pooled"][b, :nd], w["mask_pooled"][:nd]), (rep, b)
            assert not out["rois"][b, k:].any() and not out["detections"][b, nd:].any(), (rep, b)


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
def test_batched_proposals_launch_each_stage_once():
    """B = 1 and B = 8 launch the same kernels the same number of times, except the dense NMS fallback, which is
    launched once per image (mask + scan at K = 6000) and returns at once where the sparse pass succeeded."""
    from sln_amodal_b200 import ops
    c = {}
    for B in (1, 8):
        probs, deltas, anchors = _batch(261888, B, 300)
        P, D, An = cuda(probs), cuda(deltas), cuda(anchors)
        c[B] = _kernel_counts(lambda: ops.proposal_batched_device(P, D, An, 1000, 0.7, STD, HW))
    dense = {k for k in c[1] if "nms_mask_kernel" in k or "nms_scan_kernel" in k}
    assert len(dense) == 2, c[1]
    for k in dense:
        assert c[1][k] == 1 and c[8][k] == 8, (k, c[1][k], c[8].get(k))
    rest1 = {k: v for k, v in c[1].items() if k not in dense}
    rest8 = {k: v for k, v in c[8].items() if k not in dense}
    assert rest1 == rest8 and all(v == 1 for v in rest1.values()), (rest1, rest8)
    assert len(rest1) == 11, rest1                  # 5 select, rank, decode, bin, pairs, resolve, finalize


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
    A = 64
    p, d, a = torch.rand(2, A, 2), torch.rand(2, A, 4), torch.rand(A, 4)
    dets, cls = torch.rand(2, 10, 5), torch.ones(2, 10, dtype=torch.int32)
    prop = lambda *x, **kw: ops.proposal_batched_device(*x, STD, HW, **kw)
    return {
        "probs / deltas B": lambda: prop(p, torch.rand(3, A, 4), a, 10, 0.7),
        "deltas A": lambda: prop(p, torch.rand(2, A + 1, 4), a, 10, 0.7),
        "anchors A": lambda: prop(p, d, torch.rand(A - 1, 4), 10, 0.7),
        "2-D probs": lambda: prop(p[0], d, a, 10, 0.7),
        "probs last dim": lambda: prop(torch.rand(2, A, 3), d, a, 10, 0.7),
        "negative proposal_count": lambda: prop(p, d, a, -1, 0.7),
        "negative pre_nms_limit": lambda: prop(p, d, a, 10, 0.7, pre_nms_limit=-5),
        "topk 2-D dets": lambda: ops.refine_topk_batched_device(dets[0], cls, 5),
        "topk class_ids B": lambda: ops.refine_topk_batched_device(dets, torch.ones(3, 10, dtype=torch.int32), 5),
        "topk class_ids N": lambda: ops.refine_topk_batched_device(dets, torch.ones(2, 9, dtype=torch.int32), 5),
        "topk negative max_keep": lambda: ops.refine_topk_batched_device(dets, cls, -1),
    }


def test_batched_shape_mismatches_raise_without_gpu(cpu_ops):
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


def test_proposal_layer_batched_leaves_inputs_alone_without_gpu(cpu_ops, monkeypatch):
    """proposal_layer_batched hands the [B,A,*] tensors to the ops layer as they are and does not rebind `inputs`
    (the single-image drop-in squeezes them in place, like the reference)."""
    from sln_amodal_b200 import proposal
    seen = {}
    monkeypatch.setattr(proposal.ops, "proposal_batched_device",
                        lambda p, d, a, *rest, **kw: seen.update(p=p, d=d, rest=rest, kw=kw) or ("boxes", "num"))
    p, d = torch.rand(2, 64, 2), torch.rand(2, 64, 4)
    inputs = [p, d]
    out = proposal.proposal_layer_batched(inputs, 100, 0.7, torch.rand(64, 4), _GraphCfg())
    assert out == ("boxes", "num") and inputs[0] is p and inputs[1] is d and seen["p"] is p and seen["d"] is d
    assert seen["kw"]["pre_nms_limit"] == proposal.PRE_NMS_LIMIT and seen["rest"][0] == 100
