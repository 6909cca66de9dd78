"""BASELINE config 1 through the reference's own code: replay of tests/golden/predict_trace.npz.

The fixture (tests/golden/make_golden_predict.py) was recorded from the reference's unmodified
MaskRCNN.predict(mode='inference') (model.py:516-706, built as amodal_test.py:27-38 builds it; CPU, random init, one
synthetic 1024x1024 image): every call across the boundaries of the hot path with its arguments and its result --
nms, CropAndResizeFunction, proposal_layer, pyramid_roi_align, pyramid_roi_align_image, refine_detections.  Here the
same arguments go through (a) the oracle (CPU) and (b) the drop-in operators on the GPU.  The crop and pyramid calls
are stored as a seeded sample of their rows, the RPN outputs as the anchors that decide proposal_layer's result
(make_golden_predict.shrink).
"""
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import oracle
from sln_amodal_b200 import synth

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = "/root/reference"


class Trace:
    def __init__(self):
        self.g = np.load(os.path.join(HERE, "golden", "predict_trace.npz"))

    def __getitem__(self, k):
        call, _, what = k.partition("_")
        if call.startswith("proposal") and what in ("probs", "deltas"):
            return self.rpn_outputs(call)[what == "deltas"]
        a = self.g[k]
        if a.dtype.kind == "U" and a.shape == () and str(a).startswith("blob_"):
            return self.g[str(a)]
        return a

    def rpn_outputs(self, call):
        """The recorded RPN outputs [1, A, 2] / [1, A, 4] of a proposal_layer call, rebuilt from the stored top anchors
        (make_golden_predict.shrink): every other anchor scores below all of them (seeded) and has zero deltas.  The
        background column is 1 - foreground: proposal_layer reads the foreground column only."""
        top, fg = self[call + "_top"], self[call + "_top_fg"]
        n = int(self[call + "_n_anchors"])
        below = np.nextafter(fg.min(), np.float32(0))
        scores = (np.random.default_rng(0).random(n) * float(below)).astype(np.float32)
        scores[top] = fg
        deltas = np.zeros((n, 4), np.float32)
        deltas[top] = self[call + "_top_deltas"]
        return np.stack([np.float32(1) - scores, scores], 1)[None], deltas[None]

    def n(self, what):
        return int(self.g["n_" + what])


@pytest.fixture(scope="module")
def tr():
    return Trace()


def anchors_of(tr, i=0):
    """The reference's anchor pyramid is rebuilt (261 888 x 4) and checked against what the recorded run used."""
    an = synth.pyramid_anchors().astype(np.float32)
    assert tuple(tr["proposal%d_anchors_shape" % i]) == an.shape
    assert np.array_equal(an[:64], tr["proposal%d_anchors_head" % i])
    np.testing.assert_allclose(an.astype(np.float64).sum(0), tr["proposal%d_anchor_sum" % i], rtol=1e-12)
    return an


class Cfg:
    RPN_BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
    BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
    IMAGE_SHAPE = np.array([1024, 1024, 3])
    GPU_COUNT = 1
    USE_NMS = False                       # config.py:78, what the recorded run used
    DETECTION_MIN_CONFIDENCE = 0
    DETECTION_NMS_THRESHOLD = 0.3


def test_trace_covers_the_boundaries(tr):
    assert tr.n("nms") == 1 and tr.n("proposal") == 1 and tr.n("pyramid") == 2 and tr.n("refine") == 1
    assert tr.n("crop") >= 4 and tr.n("pyramid_image") == 1
    assert not bool(tr["use_nms"]) and not bool(tr["refine0_use_nms"])
    assert tr["final_detections"].shape == (1, 100, 6)


def _check_proposal_against_the_recorded_run(tr, run, exact):
    """proposal_layer (Functions.py:114-178) on the recorded RPN outputs.  The run's foreground scores contain a few
    dozen exact ties inside the top 6000 (float32 softmax), and torch's sort -- which the reference uses, :144-149 --
    leaves their order unspecified, so the reference's result is pinned in pieces that do not depend on it:
      * the cut at 6000 is clean, so the SET of decoded + clipped top-6000 boxes is unique: the recorded nms() input
        (the reference's own decode, in its own order) must equal ours as a set, bit for bit;
      * the rest of the reference's function on that input is keep = nms(dets, 0.7)[:1000] and a division by the image
        size: the recorded output must be exactly that (the nms() replay pins the keep list itself);
      * `run` (the implementation under test, ties broken by anchor index) must agree with the oracle."""
    an = anchors_of(tr)
    p, d = tr["proposal0_probs"], tr["proposal0_deltas"]
    cnt, thr = int(tr["proposal0_count"]), float(tr["proposal0_thresh"])
    fg = p[0, :, 1]
    srt = np.sort(fg)[::-1]
    assert srt[5999] > srt[6000]                                         # clean cut
    top = np.nonzero(fg >= srt[5999])[0]
    assert top.size == 6000
    boxes = oracle.clip_boxes(oracle.apply_box_deltas(an[top], d[0][top] * np.array([0.1, 0.1, 0.2, 0.2], np.float32)),
                              (0, 0, 1024, 1024))
    ours = np.concatenate([boxes, fg[top, None]], 1).astype(np.float32)
    rec = tr["nms0_dets"]
    key = lambda a: a[np.lexsort(a.T[::-1])]
    assert key(ours).tobytes() == key(rec).tobytes()
    keep = tr["nms0_keep"][:cnt]
    assert (rec[keep, :4] / np.float32(1024.0)).tobytes() == tr["proposal0_out"][0].tobytes()
    want = oracle.proposal_layer(p[0], d[0], an, cnt, thr)
    got = run(p, d, an, cnt, thr)
    assert got.shape == want.shape
    if exact:
        assert got.tobytes() == want.tobytes()
    else:
        np.testing.assert_allclose(got, want, rtol=3e-7, atol=1e-7)
    # and the tie order barely matters here: the two results share almost all of their boxes
    a = {tuple(r) for r in np.round(want, 5)}
    b = {tuple(r) for r in np.round(tr["proposal0_out"][0], 5)}
    assert len(a & b) >= 0.95 * max(len(a), len(b))


# ------------------------------------------------------------------ oracle on the recorded boundary data (CPU)
def test_oracle_replays_the_recorded_run(tr):
    d, keep = tr["nms0_dets"], tr["nms0_keep"]
    assert d.shape == (6000, 5)
    assert np.array_equal(oracle.nms(d, float(tr["nms0_thresh"])), keep)
    for i in range(tr.n("crop")):
        ph, pw = (int(v) for v in tr["crop%d_size" % i])
        got = oracle.crop_and_resize_fwd(tr["crop%d_image" % i], tr["crop%d_boxes" % i], tr["crop%d_ind" % i], ph, pw,
                                         float(tr["crop%d_ext" % i]))
        assert got.tobytes() == tr["crop%d_out" % i].tobytes()
    _check_proposal_against_the_recorded_run(tr, lambda p, d, an, cnt, thr: oracle.proposal_layer(p[0], d[0], an, cnt, thr), exact=True)
    det, keep = oracle.refine_detections(tr["refine0_rois"], tr["refine0_probs"], tr["refine0_deltas"], tr["refine0_window"],
                                         use_nms=False)
    assert np.array_equal(keep, tr["refine0_keep"]) and det.tobytes() == tr["refine0_det"].tobytes()
    for i in range(tr.n("pyramid")):
        maps = [tr["pyramid%d_map%d" % (i, l)] for l in range(int(tr["pyramid%d_nmaps" % i]))]
        got = oracle.pyramid_roi_align(tr["pyramid%d_rois" % i][0], maps, int(tr["pyramid%d_pool" % i]),
                                       tuple(int(v) for v in tr["pyramid%d_shape" % i][:2]))
        assert got.tobytes() == tr["pyramid%d_out" % i].tobytes()


# ------------------------------------------------------------------ the drop-in operators on the recorded data (GPU)
def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.gpu
def test_gpu_replays_the_recorded_run(tr):
    from nms.nms_wrapper import nms
    from roialign.roi_align.crop_and_resize import CropAndResizeFunction
    from sln_amodal_b200 import proposal_layer, pyramid_roi_align, pyramid_roi_align_image, refine_detections
    # nms(dets, thresh) at Functions.py:165: 6000 decoded RPN boxes
    keep = nms(cuda(tr["nms0_dets"]), float(tr["nms0_thresh"]))
    assert np.array_equal(keep.cpu().numpy(), tr["nms0_keep"])
    # every CropAndResizeFunction call of the run (modals.py:96,154), NCHW like the reference's tensors and channels_last
    for i in range(tr.n("crop")):
        ph, pw = (int(v) for v in tr["crop%d_size" % i])
        for cl in (False, True):
            img = cuda(tr["crop%d_image" % i])
            if cl:
                img = img.contiguous(memory_format=torch.channels_last)
            out = CropAndResizeFunction(ph, pw, float(tr["crop%d_ext" % i]))(img, cuda(tr["crop%d_boxes" % i]), cuda(tr["crop%d_ind" % i]))
            assert out.contiguous().cpu().numpy().tobytes() == tr["crop%d_out" % i].tobytes(), ("crop", i, cl)
    # proposal_layer (model.py:570): 261 888 anchors -> 6000 -> NMS 0.7 -> 1000
    _check_proposal_against_the_recorded_run(
        tr, lambda p, d, an, cnt, thr: proposal_layer([cuda(p), cuda(d)], cnt, thr, cuda(an), Cfg())[0].cpu().numpy(), exact=False)
    # refine_detections on the reference's default branch (Functions.py:526-546)
    det, keep = refine_detections(cuda(tr["refine0_rois"]), cuda(tr["refine0_probs"]), cuda(tr["refine0_deltas"]),
                                  tuple(float(v) for v in tr["refine0_window"]), Cfg())
    assert np.array_equal(keep.cpu().numpy(), tr["refine0_keep"])
    assert det.cpu().numpy().tobytes() == tr["refine0_det"].tobytes()
    # pyramid_roi_align (modals.py:20-110) for the classifier (7x7) and the mask head (16x16), pyramid_roi_align_image
    for i in range(tr.n("pyramid")):
        maps = [cuda(tr["pyramid%d_map%d" % (i, l)]) for l in range(int(tr["pyramid%d_nmaps" % i]))]
        got = pyramid_roi_align([cuda(tr["pyramid%d_rois" % i])] + maps, int(tr["pyramid%d_pool" % i]),
                                tuple(int(v) for v in tr["pyramid%d_shape" % i]))
        assert got.contiguous().cpu().numpy().tobytes() == tr["pyramid%d_out" % i].tobytes(), ("pyramid", i)
    got = pyramid_roi_align_image([cuda(tr["pyrimg0_rois"]), cuda(tr["pyrimg0_map"])], int(tr["pyrimg0_pool"]),
                                  tuple(int(v) for v in tr["pyrimg0_shape"]))
    assert got.contiguous().cpu().numpy().tobytes() == tr["pyrimg0_out"].tobytes()


# ------------------------------------------------------------------ the real reference modules pick the drop-ins up (CPU)
@pytest.mark.skipif(not os.path.isdir(REF), reason="needs the reference checkout (build container only)")
def test_install_rebinds_the_real_reference_modules():
    """Imports the REAL model.py / modal/Functions.py / modal/modals.py from /root/reference with THIS repo ahead of it on
    sys.path (third-party imports the container lacks are stubbed): the reference's own import statements resolve to the
    shadow packages, and install() rebinds the names the reference looks up at call time."""
    code = r'''
import sys, types
sys.path.insert(0, %r)
sys.path.append(%r)
def stub(name, **kw):
    m = types.ModuleType(name); m.__dict__.update(kw); sys.modules[name] = m; return m
cm = stub("matplotlib.cm"); stub("matplotlib", cm=cm, use=lambda *a, **k: None)
for n in ("matplotlib.pyplot", "matplotlib.patches", "matplotlib.lines", "skimage", "skimage.color", "skimage.io",
          "skimage.morphology", "skimage.transform"):
    stub(n)
stub("skimage.measure", label=None, regionprops=None)
stub("tensorboardX", SummaryWriter=lambda *a, **k: None)
import model, modal.Functions as F, modal.modals as M
import sln_amodal_b200 as S
from sln_amodal_b200 import crop_and_resize, proposal, pyramid, detection, targets
snms = sys.modules['sln_amodal_b200.nms']
# the reference's own import lines (modals.py:6, Functions.py:5,7) resolved to this repo's shadows
assert M.CropAndResizeFunction is crop_and_resize.CropAndResizeFunction, M.CropAndResizeFunction
assert F.CropAndResizeFunction is crop_and_resize.CropAndResizeFunction
assert F.nms is snms.nms, F.nms
assert "/root/reference" in model.__file__ and "/root/reference" in F.__file__
done = S.install()
assert model.proposal_layer is proposal.proposal_layer and F.proposal_layer is proposal.proposal_layer
assert M.pyramid_roi_align is pyramid.pyramid_roi_align
assert model.pyramid_roi_align_image is pyramid.pyramid_roi_align_image
assert model.refine_detections is detection.refine_detections and F.refine_detections is detection.refine_detections
assert model.detection_target_layer is targets.detection_target_layer
assert "model.MaskRCNN.unmold_detections" in done
# detection_layer (Functions.py:560) is the reference's own; it finds refine_detections in its module globals at call time
assert F.detection_layer.__globals__["refine_detections"] is detection.refine_detections
print("ok", len(done))
''' % (ROOT, REF)
    import subprocess
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip().startswith("ok"), r.stdout + r.stderr[-2000:]
