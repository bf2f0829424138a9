"""Pin the oracle (CPU only): against every golden vector the reference's own tests hold for this path, against what the
reference's C++ CPU kernels return (compiled by oracle/build_ref.py; results stored in tests/golden/mmcv_cpu_ops_ref.pt by
tests/golden/make_mmcv_ops_golden.py), and against the committed model-level fixtures under tests/golden/.  No GPU, no
compute through the C ABI."""
import json
import os

import numpy as np
import pytest
import torch
import torchvision

from oracle import ops as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def ref():
    return torch.load(os.path.join(GOLD, "mmcv_cpu_ops_ref.pt"))


# ---------------------------------------------------------------- reference golden vectors
def test_nms_golden_vectors():
    # mmcv/tests/test_ops/test_nms.py:13-20
    b = np.array([[6.0, 3.0, 8.0, 7.0], [3.0, 6.0, 9.0, 11.0], [3.0, 7.0, 10.0, 12.0], [1.0, 4.0, 13.0, 7.0]], dtype=np.float32)
    s = np.array([0.6, 0.9, 0.7, 0.2], dtype=np.float32)
    for form in ("cuda", "cpu"):
        assert O.nms_ref(b, s, 0.3, iou_form=form).tolist() == [1, 0, 3]
    # mmcv/mmcv/ops/nms.py:139-150 (docstring example: 3 kept)
    boxes = np.array([[49.1, 32.4, 51.0, 35.9], [49.3, 32.9, 51.0, 35.3], [49.2, 31.8, 51.0, 35.4], [35.1, 11.5, 39.1, 15.7],
                      [35.6, 11.8, 39.3, 14.2], [35.3, 11.5, 39.9, 14.5], [35.2, 11.7, 39.7, 15.7]], dtype=np.float32)
    scores = np.array([0.9, 0.9, 0.5, 0.5, 0.5, 0.4, 0.3], dtype=np.float32)
    assert len(O.nms_ref(boxes, scores, 0.6)) == 3


ROI_INPUTS = [([[[[1., 2.], [3., 4.]]]], [[0., 0., 0., 1., 1.]]),
              ([[[[1., 2.], [3., 4.]], [[4., 3.], [2., 1.]]]], [[0., 0., 0., 1., 1.]]),
              ([[[[1., 2., 5., 6.], [3., 4., 7., 8.], [9., 10., 13., 14.], [11., 12., 15., 16.]]]], [[0., 0., 0., 3., 3.]])]
ROI_OUTPUTS = [[[[[1.0, 1.25], [1.5, 1.75]]]], [[[[1.0, 1.25], [1.5, 1.75]], [[4.0, 3.75], [3.5, 3.25]]]],
               [[[[1.9375, 4.75], [7.5625, 10.375]]]]]


def test_roi_align_golden_vectors():
    # mmcv/tests/test_ops/test_roi_align.py:14-32,67-104 (forward values; pool 2x2, scale 1, sampling 2, avg, aligned)
    for (inp, rois), want in zip(ROI_INPUTS, ROI_OUTPUTS):
        got = O.roi_align_ref(torch.tensor(inp), torch.tensor(rois), 2, 1.0, 2, True)
        assert np.allclose(got.numpy(), np.array(want), atol=1e-6)


def test_msda_equivalence_setup():
    # the configuration of mmcv/tests/test_ops/test_ms_deformable_attn.py:73-135 (seed 3, N=1,M=2,D=2,Lq=2,L=2,P=2):
    # our restatement must agree with a direct per-sample bilinear evaluation (the CUDA kernel's definition)
    torch.manual_seed(3)
    N, M, D, Lq, L, P = 1, 2, 2, 2, 2, 2
    shapes = [(6, 4), (3, 2)]
    S = sum(h * w for h, w in shapes)
    value = torch.rand(N, S, M, D) * 0.01
    loc = torch.rand(N, Lq, M, L, P, 2)
    aw = torch.rand(N, Lq, M, L, P) + 1e-5
    aw = aw / aw.sum(-1, keepdim=True).sum(-2, keepdim=True)
    got = O.msda_ref(value, shapes, loc, aw)
    want = torch.zeros(N, Lq, M * D)
    starts = [0, shapes[0][0] * shapes[0][1]]
    for q in range(Lq):
        for m in range(M):
            for l, (H, W) in enumerate(shapes):
                for p in range(P):
                    x, y = loc[0, q, m, l, p, 0] * W - 0.5, loc[0, q, m, l, p, 1] * H - 0.5
                    x0, y0 = int(np.floor(x)), int(np.floor(y))
                    for dy in (0, 1):
                        for dx in (0, 1):
                            xx, yy = x0 + dx, y0 + dy
                            if 0 <= xx < W and 0 <= yy < H:
                                wgt = (1 - abs(x - xx)) * (1 - abs(y - yy))
                                want[0, q, m * D:(m + 1) * D] += aw[0, q, m, l, p] * wgt * value[0, starts[l] + yy * W + xx, m]
    assert (got - want).abs().max() < 1e-9 + 1e-6 * want.abs().max()


# ---------------------------------------------------------------- the reference's own compiled CPU kernels
def test_nms_matches_compiled_reference(ref):
    assert len(ref["nms_cases"]) == 4
    for case, want_by_thr in zip(ref["nms_cases"], ref["nms"]):
        boxes, scores = case["boxes"], case["scores"]
        for thr in (0.3, 0.6):
            want = want_by_thr[thr]
            got = O.nms_ref(boxes.numpy(), scores.numpy(), thr, 0, iou_form="cpu")
            assert got.tolist() == want.tolist()
            # the CUDA-form inequality (what the GPU path implements) selects the same boxes on these inputs
            assert O.nms_ref(boxes.numpy(), scores.numpy(), thr, 0, iou_form="cuda").tolist() == want.tolist()
    assert ref["nms_empty_numel"] == 0


def test_roi_align_matches_compiled_reference(ref):
    x, rois = ref["roi_x"], ref["roi_rois"]
    assert [r["scale"] for r in ref["roi"]] == [8 / 14, 4 / 14, 2 / 14]
    for r in ref["roi"]:            # a fixed sample of each 30 x 5 x 14 x 14 output
        got = O.roi_align_ref(x, rois, 14, r["scale"], 2, True)
        assert (got.reshape(-1)[r["index"].long()] - r["values"]).abs().max() < 1e-5


def test_reference_cpu_roi_align_rejects_negative_extents(ref):
    # SURVEY T2: the literal reference CPU path raises on the cxcywh-as-xyxy boxes Groma feeds it; the oracle follows the
    # CUDA kernel instead (same as torchvision's CPU roi_align), which is finite there.
    x = torch.randn(1, 3, 32, 32)
    rois = torch.tensor([[0.0, 200.0, 200.0, 50.0, 50.0]])
    assert "non-negative size" in ref["negative_extent_error"]     # the reference kernel raised on these rois
    got = O.roi_align_ref(x, rois, 14, 8 / 14, 2, True)
    tv = torchvision.ops.roi_align(x, rois, 14, 8 / 14, 2, True)
    assert torch.isfinite(got).all() and (got - tv).abs().max() < 1e-6


# ---------------------------------------------------------------- committed model-level fixtures
def test_oracle_reproduces_golden_fixture(tmp_path):
    from tests.golden import make_golden
    path = os.path.join(GOLD, "tiny_forward.pt")
    if not os.path.exists(path):
        pytest.skip("fixture missing")
    gold = torch.load(path)
    out = make_golden.run_canonical(str(tmp_path / "oracle.pt"))     # the fixture's CPU settings, so the same bits on any CPU
    assert torch.equal(out["input_ids"], gold["input_ids"])
    assert torch.equal(out["new_tokens"], gold["new_tokens"])
    assert [x.tolist() for x in out["nms_inds"]] == [x.tolist() for x in gold["nms_inds"]]
    assert (out["pred_boxes"] - gold["pred_boxes"]).abs().max() < 1e-5
    assert (out["last_logits"] - gold["last_logits"]).abs().max() < 1e-4 * gold["last_logits"].abs().max()
