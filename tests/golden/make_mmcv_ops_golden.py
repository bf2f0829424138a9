"""Generate tests/golden/mmcv_cpu_ops_ref.pt: what the REFERENCE's own mmcv C++ CPU kernels for `nms` and `roi_align_forward`
return on the inputs of tests/test_oracle_pinned.py.  The kernels are compiled from the reference sources where they lie by
oracle/build_ref.py (nothing is copied into the repo); the reference is not part of this repository, hence the committed
fixture.   python -m tests.golden.make_mmcv_ops_golden

RoIAlign outputs are stored as a fixed sample (seed 0, ROI_SAMPLE elements per scale, flat indices stored beside them) to keep
the file small."""
import os

import torch

from oracle import build_ref

HERE = os.path.dirname(os.path.abspath(__file__))
ROI_SCALES = (8 / 14, 4 / 14, 2 / 14)
ROI_SAMPLE = 2048


def nms_cases():
    g = torch.Generator().manual_seed(0)
    out = []
    for n in (1, 7, 64, 300):
        ctr = torch.rand(n, 2, generator=g); wh = torch.rand(n, 2, generator=g) * 0.3 + 0.02
        if n > 20:
            ctr[n // 2:] = ctr[:n - n // 2] + 0.01 * torch.randn(n - n // 2, 2, generator=g)
            wh[n // 2:] = wh[:n - n // 2]
        boxes = torch.cat([ctr - wh / 2, ctr + wh / 2], -1).contiguous()
        scores = torch.rand(n, generator=g)
        out.append(dict(boxes=boxes, scores=scores))
    return out


def roi_case():
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 5, 32, 32, generator=g)
    rois = torch.rand(30, 5, generator=g) * 300
    rois[:, 0] = torch.randint(0, 2, (30,), generator=g).float()
    rois[:, 3:] = rois[:, 1:3] + torch.rand(30, 2, generator=g) * 120   # non-negative extents: the CPU kernel asserts on negative
    return x, rois


def negative_extent_case():
    x = torch.randn(1, 3, 32, 32, generator=torch.Generator().manual_seed(2))
    rois = torch.tensor([[0.0, 200.0, 200.0, 50.0, 50.0]])
    return x, rois


def run_reference():
    ref = build_ref.load_ref()
    if ref is None:
        raise RuntimeError("oracle/_ref is not built and the reference sources are absent (python -m oracle.build_ref)")
    nms = []
    for c in nms_cases():
        nms.append({thr: ref.nms(c["boxes"], c["scores"], thr, 0) for thr in (0.3, 0.6)})
    empty = ref.nms(torch.zeros(0, 4), torch.zeros(0), 0.5, 0).numel()
    x, rois = roi_case()
    roi = []
    for k, scale in enumerate(ROI_SCALES):
        out = torch.zeros(30, 5, 14, 14)
        ref.roi_align_forward(x, rois, out, torch.zeros(0), torch.zeros(0), 14, 14, scale, 2, 1, True)
        idx = torch.randperm(out.numel(), generator=torch.Generator().manual_seed(k))[:ROI_SAMPLE].sort().values
        roi.append(dict(scale=scale, index=idx.to(torch.int32), values=out.reshape(-1)[idx].clone()))
    xn, rn = negative_extent_case()
    try:
        ref.roi_align_forward(xn, rn, torch.zeros(1, 3, 14, 14), torch.zeros(0), torch.zeros(0), 14, 14, 8 / 14, 2, 1, True)
        negative = ""
    except Exception as e:
        negative = str(e).splitlines()[0].rsplit(". ", 1)[-1]      # the kernel's own message, without the source location
    return dict(nms_cases=nms_cases(), nms=nms, nms_empty_numel=empty, roi_x=x, roi_rois=rois, roi=roi,
                negative_extent_error=negative)


if __name__ == "__main__":
    out = run_reference()
    torch.save(out, os.path.join(HERE, "mmcv_cpu_ops_ref.pt"))
    print("wrote mmcv_cpu_ops_ref.pt; negative-extent RoI:", out["negative_extent_error"] or "no error")
