"""detection_target_layer_batched against the single-image detection_target_layer, the golden vectors and the oracle.

Every image of a batched call is compared with detection_target_layer on that image alone under the same seed, bit for
bit (torch.equal), together with the CPU generator's state afterwards.  The golden and oracle comparisons hold the
batched path to the reference directly, including the one rule where it follows the reference and the single-image path
does not (a proposal whose IoU maximum is NaN).  The input-contract tests at the end run without a device, against a
stub of the library that fails when it is called.
"""
import contextlib
import os

import numpy as np
import pytest
import torch

from oracle import oracle
from sln_amodal_b200 import synth

gpu = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class Cfg:
    BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
    TRAIN_ROIS_PER_IMAGE = 100
    ROI_POSITIVE_RATIO = 0.7
    MASK_SHAPE = [32, 32]
    USE_MINI_MASK = False


class MiniCfg(Cfg):
    USE_MINI_MASK = True


def dev():
    return torch.device("cuda", 0)


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev())


# bench.py detection_targets_metric's generator, one seed per image; `kind` makes the edge cases
def _image(seed, kind="plain", G=12, N=1000, L=1, S=1024):
    rng = np.random.default_rng(seed)
    gt = np.zeros((G, 4), np.float32)
    masks = np.zeros((L, G, S, S), np.uint8)
    lo, hi = (0.0, 0.45) if kind == "no_pos" else (0.0, 1.0)
    for i in range(G):
        h, w = rng.uniform(0.1, 0.4, 2) * (hi - lo)
        y1, x1 = lo + rng.uniform(0, hi - lo - h), lo + rng.uniform(0, hi - lo - w)
        gt[i] = (y1, x1, y1 + h, x1 + w)
        for l in range(L):                                    # layer l: the top (1 - l/4) of the box
            masks[l, i, int(y1 * S):int((y1 + h * (1 - l / 4)) * S), int(x1 * S):int((x1 + w) * S)] = 1
    jit = gt[rng.integers(0, G, 240)] + rng.normal(0, 0.02, (240, 4)).astype(np.float32)
    props = np.clip(np.concatenate([jit, synth.roi_boxes(N - 240, seed=seed % 997)], 0), 0, 1).astype(np.float32)
    ids = np.ones(G, np.int32)
    if kind == "no_pos":                                      # GT boxes in [0, 0.45]^2, proposals in [0.55, 1]^2
        props = (0.55 + 0.45 * synth.roi_boxes(N, seed=seed % 997)).astype(np.float32)
    elif kind == "no_neg":                                    # every proposal is one of the first 8 GT boxes: no
        props = gt[rng.integers(0, 8, N)].copy()              # eligible negative (num_gt >= 9 in the ragged test)
    elif kind == "crowd":                                     # a crowd row and a class-0 row
        ids[1], ids[4] = -1, 0
    return props, ids, gt, masks


def _batch(kinds, seed, G=12, N=1000, L=1, S=1024):
    imgs = [_image(seed + 31 * b, k, G, N, L, S) for b, k in enumerate(kinds)]
    return [np.stack([im[j] for im in imgs]) for j in range(4)]


def _run_and_compare(props, ids, gt, masks, cfg, seed, num_proposals=None, num_gt=None, as_list=False, as_bool=False):
    """One batched call and B single-image calls under the same seed; every image and the generator state compared."""
    from sln_amodal_b200 import detection_target_layer, detection_target_layer_batched
    B, R, G = props.shape[0], props.shape[1], gt.shape[1]
    P, I, Gb = cuda(props), cuda(ids), cuda(gt)
    M = cuda(masks)
    if as_bool:
        M = M.bool()
    ng = [G] * B if num_gt is None else list(num_gt)
    npr = [R] * B if num_proposals is None else [int(v) for v in num_proposals]
    Mb = [M[b][:, :ng[b]] for b in range(B)] if as_list else M
    NP = None if num_proposals is None else torch.tensor(npr, dtype=torch.int32, device=dev())
    torch.manual_seed(seed)
    rois, cls, deltas, tm, n_pos, n_rois = detection_target_layer_batched(P, I, Gb, Mb, cfg, num_proposals=NP,
                                                                          num_gt=num_gt)
    state = torch.get_rng_state()
    T = rois.shape[1]
    L = masks.shape[1]
    assert rois.shape == (B, T, 4) and cls.shape == (B, T) and deltas.shape == (B, T, 4)
    assert tm.shape == (B, T, L) + tuple(cfg.MASK_SHAPE) and cls.dtype == torch.int32
    assert n_pos.dtype == torch.int32 and n_rois.dtype == torch.int32 and n_pos.shape == (B,) and n_rois.shape == (B,)
    torch.manual_seed(seed)
    counts = []
    for b in range(B):
        r, c, d, m = detection_target_layer(P[b, :npr[b]].unsqueeze(0), I[b, :ng[b]].unsqueeze(0), Gb[b, :ng[b]].unsqueeze(0),
                                            M[b][:, :ng[b]].unsqueeze(0), cfg)
        k, p = int(n_rois[b]), int(n_pos[b])
        counts.append((p, k))
        if r.numel() == 0:
            assert k == 0 and p == 0, b
        else:
            assert k == r.shape[0], b
            assert torch.equal(rois[b, :k], r), b
            assert torch.equal(cls[b, :k], c), b
            assert torch.equal(deltas[b, :k], d), b
            assert torch.equal(tm[b, :k], m), b
            assert not cls[b, p:k].any() and not deltas[b, p:k].any() and not tm[b, p:k].any(), b
        assert not rois[b, k:].any() and not cls[b, k:].any() and not deltas[b, k:].any() and not tm[b, k:].any(), b
    assert torch.equal(torch.get_rng_state(), state)
    return counts


def _garbage_pads(props, ids, gt, npr, ng):
    """Rows past num_proposals / num_gt that would change the result if they were read: proposals on top of GT boxes,
    GT rows on top of proposals with a crowd class."""
    for b in range(props.shape[0]):
        props[b, npr[b]:] = gt[b, np.arange(props.shape[1] - npr[b]) % gt.shape[1]]
        gt[b, ng[b]:] = props[b, :gt.shape[1] - ng[b]]
        ids[b, ng[b]:] = -1


KINDS = ["plain", "no_pos", "no_neg", "crowd", "plain"]


@gpu
@pytest.mark.parametrize("B", [1, 2, 5, 16])
def test_batched_targets_equal_single_image_targets(B):
    """Edge cases by image: no positive, no eligible negative, crowd + class-0 rows, ragged num_proposals / num_gt
    (padding that would be matched if read), stacked u8 masks and a list of bool masks."""
    kinds = [KINDS[b % len(KINDS)] for b in range(B)]
    props, ids, gt, masks = _batch(kinds, 1000 + B)
    R, G = props.shape[1], gt.shape[1]
    npr = [R - (137 * b) % 400 for b in range(B)]
    ng = [G - (b % 4) for b in range(B)]
    _garbage_pads(props, ids, gt, npr, ng)
    counts = _run_and_compare(props, ids, gt, masks, Cfg(), seed=7 + B, num_proposals=npr, num_gt=ng)
    if B >= 5:
        assert counts[1] == (0, 0)                            # no_pos
        assert counts[2][0] > 0 and counts[2][1] == counts[2][0]   # no_neg: positives only
        assert counts[0][1] == 100 and counts[3][0] > 0       # plain fills T; crowd samples
    _run_and_compare(props, ids, gt, masks, Cfg(), seed=8 + B, num_proposals=npr, num_gt=ng, as_list=True, as_bool=True)


@gpu
@pytest.mark.parametrize("L", [1, 3])
def test_batched_targets_mini_mask_and_layers(L):
    """USE_MINI_MASK = True (the positives' boxes in their GT box's frame), L layers, list and stacked masks, defaults
    for num_proposals / num_gt."""
    props, ids, gt, masks = _batch(["plain", "crowd", "no_neg"], 50 + L, L=L, S=512)
    for cfg in (Cfg(), MiniCfg()):
        _run_and_compare(props, ids, gt, masks, cfg, seed=L)
        _run_and_compare(props, ids, gt, masks, cfg, seed=L + 10, as_list=True, as_bool=L == 3)


@gpu
def test_batched_targets_take_proposal_layer_batched_output():
    """proposal_layer_batched's rois [B,1000,4] (zero padded) and num [B] go straight in."""
    from sln_amodal_b200 import detection_target_layer_batched, ops
    B, A = 4, 261888
    rng = np.random.default_rng(5)
    anchors = synth.pyramid_anchors().astype(np.float32)
    fg = rng.uniform(0, 1, (B, A)).astype(np.float32)
    probs = np.stack([1 - fg, fg], 2)
    deltas = (rng.standard_normal((B, A, 4)) * 0.5).astype(np.float32)
    rois, num = ops.proposal_batched_device(cuda(probs), cuda(deltas), cuda(anchors), 1000, 0.7, (0.1, 0.1, 0.2, 0.2),
                                            (1024, 1024))
    n_h = num.cpu().numpy()
    r_h = rois.cpu().numpy()
    _, ids, gt, masks = _batch(["plain"] * B, 77, S=512)
    for b in range(B):                                        # GT boxes = some of the image's proposals, jittered
        gt[b] = np.clip(r_h[b, rng.integers(0, n_h[b], gt.shape[1])] + rng.normal(0, 0.01, (gt.shape[1], 4)), 0, 1)
    _run_and_compare(r_h, ids, gt.astype(np.float32), masks, Cfg(), seed=3, num_proposals=n_h)
    # the device tensors themselves, without a host copy of the proposals
    torch.manual_seed(3)
    out = detection_target_layer_batched(rois, cuda(ids), cuda(gt.astype(np.float32)), cuda(masks), Cfg(), num_proposals=num)
    torch.manual_seed(3)
    again = detection_target_layer_batched(cuda(r_h), cuda(ids), cuda(gt.astype(np.float32)), cuda(masks), Cfg(),
                                           num_proposals=num)
    assert all(torch.equal(a, b) for a, b in zip(out, again))
    assert int(out[5].min()) > 0


# ---- the golden vectors and the oracle
def _golden_cases():
    g = np.load(os.path.join(GOLDEN, "detection_targets.npz"))
    for k in range(int(g["n_cases"])):
        shp = tuple(int(v) for v in g["masks_shape%d" % k])
        masks = np.unpackbits(g["masks%d" % k])[: int(np.prod(shp))].reshape(shp)
        tshp = tuple(int(v) for v in g["tmasks_shape%d" % k])
        n_t = int(np.prod(tshp)) if len(tshp) > 1 else 0
        tmasks = np.unpackbits(g["tmasks%d" % k])[:n_t].reshape(tshp).astype(np.float32) if n_t else np.zeros(0, np.float32)
        yield dict(props=g["props%d" % k], ids=g["ids%d" % k], gt=g["gt%d" % k], masks=masks, seed=int(g["seed%d" % k]),
                   rois=g["rois%d" % k], cls=g["cls%d" % k], deltas=g["deltas%d" % k], tmasks=tmasks)


def _pad_batch(cases):
    """Cases of different N / G as one batch: padded proposals and GT rows, the masks as a list of [L,G_b,H,W]."""
    B = len(cases)
    R = max(c["props"].shape[0] for c in cases)
    G = max(c["gt"].shape[0] for c in cases)
    props = np.zeros((B, R, 4), np.float32)
    gt = np.zeros((B, G, 4), np.float32)
    ids = np.zeros((B, G), np.int32)
    for b, c in enumerate(cases):
        props[b, :c["props"].shape[0]] = c["props"]
        gt[b, :c["gt"].shape[0]] = c["gt"]
        ids[b, :c["ids"].shape[0]] = c["ids"]
    npr = torch.tensor([c["props"].shape[0] for c in cases], dtype=torch.int32, device=dev())
    ng = [int(c["gt"].shape[0]) for c in cases]
    return cuda(props), cuda(ids), cuda(gt), [cuda(c["masks"]) for c in cases], npr, ng


def _assert_matches(out, b, rois, cls, deltas, tm):
    k = int(out[5][b])
    if rois.size == 0:
        assert k == 0
        return
    assert k == rois.shape[0]
    assert np.array_equal(out[0][b, :k].cpu().numpy(), rois) and np.array_equal(out[1][b, :k].cpu().numpy(), cls)
    np.testing.assert_allclose(out[2][b, :k].cpu().numpy(), deltas, rtol=3e-6, atol=1e-6)
    assert np.array_equal(out[3][b, :k].cpu().numpy(), tm)


@gpu
def test_batched_targets_match_golden_and_oracle():
    from sln_amodal_b200 import detection_target_layer_batched
    cases = list(_golden_cases())
    for c in cases:                                           # each case under its own stored seed: a batch of one
        P, I, Gb, M, npr, ng = _pad_batch([c])
        torch.manual_seed(c["seed"])
        out = detection_target_layer_batched(P, I, Gb, M, Cfg(), num_proposals=npr, num_gt=ng)
        _assert_matches(out, 0, c["rois"], c["cls"], c["deltas"], c["tmasks"])
    P, I, Gb, M, npr, ng = _pad_batch(cases)                  # the three as one batch, ragged G, one seed
    torch.manual_seed(11)
    out = detection_target_layer_batched(P, I, Gb, M, Cfg(), num_proposals=npr, num_gt=ng)
    torch.manual_seed(11)
    for b, c in enumerate(cases):
        _assert_matches(out, b, *oracle.detection_target_layer(c["props"], c["ids"], c["gt"], c["masks"]))


@gpu
def test_batched_targets_nan_iou_rows_follow_the_reference():
    """A zero-area proposal against a zero-area GT box has IoU 0/0 = NaN: the reference samples it neither as a positive
    nor as a negative (NaN < 0.5 is false), and so does the batched call."""
    from sln_amodal_b200 import detection_target_layer_batched
    props, ids, gt, masks = _image(9, S=256)
    gt[5] = (0.5, 0.5, 0.5, 0.5)                              # zero-area GT box
    nan_rows = np.arange(0, 1000, 7)
    props[nan_rows, 2] = props[nan_rows, 0]                   # zero-area proposals: every IoU against gt[5] is NaN
    props[nan_rows, 3] = props[nan_rows, 1]
    torch.manual_seed(4)
    out = detection_target_layer_batched(cuda(props[None]), cuda(ids[None]), cuda(gt[None]), cuda(masks[None]), Cfg())
    torch.manual_seed(4)
    want = oracle.detection_target_layer(props, ids, gt, masks)
    _assert_matches(out, 0, *want)
    k = int(out[5][0])
    sampled = out[0][0, :k].cpu().numpy()
    assert k > int(out[4][0]) > 0
    assert not (sampled[:, 0] == sampled[:, 2]).any()        # no zero-area (NaN) proposal among the sampled rows


@gpu
@pytest.mark.parametrize("B", [1, 5])
def test_batched_targets_two_launches_one_host_copy(B, monkeypatch):
    from sln_amodal_b200 import _lib, detection_target_layer_batched
    props, ids, gt, masks = _batch(["plain", "crowd", "no_pos", "no_neg", "plain"][:B], 600, S=256)
    args = (cuda(props), cuda(ids), cuda(gt), cuda(masks), Cfg())
    detection_target_layer_batched(*args)
    torch.cuda.synchronize()
    copies = []
    real_cpu = torch.Tensor.cpu

    def counting_cpu(self, *a, **kw):
        if self.is_cuda:
            copies.append(tuple(self.shape))
        return real_cpu(self, *a, **kw)

    monkeypatch.setattr(torch.Tensor, "cpu", counting_cpu)
    l0 = _lib.launches()
    detection_target_layer_batched(*args)
    assert _lib.launches() - l0 == 2
    assert copies == [(B, props.shape[1])]                   # the codes: one byte per proposal


# ---- input contract without a GPU: CPU tensors, and a library stub that fails the test when anything reaches it
class _LibStub:
    def __getattr__(self, name):
        def called(*args):
            raise AssertionError(f"{name} was called: the ops layer let the call through to the kernels")
        return called


ON_CPU = set()                                                # ids of the tensors the stubbed check treats as host tensors


@pytest.fixture
def cpu_ops(monkeypatch):
    from sln_amodal_b200 import _lib, ops

    def require_cuda(t, name):
        if id(t) in ON_CPU:
            raise _lib.SlnError(f"{name} must be a CUDA tensor")

    monkeypatch.setattr(ops, "_require_cuda", require_cuda)
    monkeypatch.setattr(ops, "lib", lambda: _LibStub())
    monkeypatch.setattr(ops, "stream_ptr", lambda: None)
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    yield ops
    ON_CPU.clear()


def _good(B=2, R=50, G=6, L=1):
    return dict(proposals=torch.rand(B, R, 4), gt_class_ids=torch.ones(B, G, dtype=torch.int32), gt_boxes=torch.rand(B, G, 4),
                gt_masks=torch.zeros(B, L, G, 16, 16, dtype=torch.uint8))


def _bad_calls():
    host_masks = torch.zeros(2, 1, 6, 16, 16, dtype=torch.uint8)
    ON_CPU.add(id(host_masks))
    return {
        "2-D proposals": dict(proposals=torch.rand(50, 4)),
        "f64 proposals": dict(proposals=torch.rand(2, 50, 4, dtype=torch.float64)),
        "gt_boxes B": dict(gt_boxes=torch.rand(3, 6, 4)),
        "f16 gt_boxes": dict(gt_boxes=torch.rand(2, 6, 4).half()),
        "gt_class_ids G": dict(gt_class_ids=torch.ones(2, 5, dtype=torch.int32)),
        "float gt_class_ids": dict(gt_class_ids=torch.ones(2, 6)),
        "num_gt > G": dict(num_gt=[3, 7]),
        "num_gt length": dict(num_gt=[3]),
        "negative num_gt": dict(num_gt=[3, -1]),
        "list entry G_b": dict(gt_masks=[torch.zeros(1, 6, 16, 16, dtype=torch.uint8), torch.zeros(1, 4, 16, 16, dtype=torch.uint8)],
                               num_gt=[6, 5]),
        "list length": dict(gt_masks=[torch.zeros(1, 6, 16, 16, dtype=torch.uint8)]),
        "list L / H / W": dict(gt_masks=[torch.zeros(1, 6, 16, 16, dtype=torch.uint8), torch.zeros(2, 6, 16, 16, dtype=torch.uint8)]),
        "stacked masks G": dict(gt_masks=torch.zeros(2, 1, 5, 16, 16, dtype=torch.uint8)),
        "4-D stacked masks": dict(gt_masks=torch.zeros(1, 6, 16, 16, dtype=torch.uint8)),
        "masks on the CPU": dict(gt_masks=host_masks),
        "float masks": dict(gt_masks=torch.zeros(2, 1, 6, 16, 16)),
        "num_proposals length": dict(num_proposals=torch.tensor([50, 40, 30], dtype=torch.int32)),
        "int64 num_proposals": dict(num_proposals=torch.tensor([50, 40])),
        "B above 512": dict(_good(B=513, R=2, G=1)),
    }


def test_batched_targets_malformed_inputs_raise_without_gpu(cpu_ops):
    from sln_amodal_b200 import _lib, detection_target_layer_batched
    missed = []
    for what, change in _bad_calls().items():
        kw = _good()
        kw.update(change)
        l0 = _lib.launches()
        try:
            detection_target_layer_batched(config=Cfg(), **kw)
            missed.append(f"{what}: no error")
        except _lib.SlnError:
            if _lib.launches() != l0:
                missed.append(f"{what}: launches counted")
        except Exception as e:                   # reached the stub, or CUDA-only code further down
            missed.append(f"{what}: {type(e).__name__}: {e}")
    assert not missed, missed


def test_batched_targets_good_inputs_reach_the_library_without_gpu(cpu_ops):
    """The checks let well-formed input through (ragged list masks, bool, num_gt / num_proposals given): the call gets
    as far as the first kernel, the stub."""
    from sln_amodal_b200 import detection_target_layer_batched
    kw = _good()
    kw.update(gt_masks=[torch.zeros(1, 6, 16, 16, dtype=torch.bool), torch.zeros(1, 4, 16, 16, dtype=torch.bool)],
              num_gt=[6, 4], num_proposals=torch.tensor([50, 20], dtype=torch.int32))
    with pytest.raises(AssertionError, match="sln_target_match_batched was called"):
        detection_target_layer_batched(config=Cfg(), **kw)


def test_rois_per_image_is_the_largest_sample():
    from sln_amodal_b200.targets import rois_per_image
    assert rois_per_image(Cfg()) == 100

    class C2(Cfg):
        TRAIN_ROIS_PER_IMAGE = 200
        ROI_POSITIVE_RATIO = 0.33

    want, r = int(200 * 0.33), 1.0 / 0.33
    assert rois_per_image(C2()) == max(p + int(r * p - p) for p in range(1, want + 1))
