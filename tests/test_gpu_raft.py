"""GPU: the ProPainter stages (SURVEY.md §8a P3-P6) on the device runtime against the oracle and the unmodified reference's frames.
Tolerance (fp16 features, fp32 flow state; the fp16 simulation of the stand-in gives EPE mean 8e-4 / max 7e-3 px on this fixture,
profiles/fp16_forecast_r1.md): mean end-point error <= 0.01 px, max <= 0.1 px."""
import os

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import raft_oracle as R
from oracle import sttn_oracle as O

PATH = os.path.join(ROOT, "weights", "propainter", "raft-things.pth")
pytestmark = pytest.mark.gpu
needs_raft = pytest.mark.skipif(not os.path.exists(PATH), reason="raft-things.pth not staged under weights/propainter")


def check_raft_flows(runtime=None):
    """the stage check itself; `runtime` = None runs on cuda:0, tests/test_stage_checks_rehearsed_cpu.py passes the hybrid CPU runtime"""
    from vsr_b200.raft_flow import RaftFlow

    frames = O.synthetic_clip(3, 128, 192, seed=23)
    ff, fb = RaftFlow(PATH, "cuda:0", runtime=runtime)(frames)
    x = torch.from_numpy(np.stack([f[:, :, ::-1] for f in frames]).astype(np.float32) / 255).permute(0, 3, 1, 2)[None] * 2 - 1
    wf, wb = R.raft_bi(R.load_weights(PATH), x)
    for got, want in ((ff, wf[0].numpy()), (fb, wb[0].numpy())):
        epe = np.sqrt(((got - want) ** 2).sum(1))
        assert np.isfinite(got).all() and epe.mean() <= 0.01 and epe.max() <= 0.1, (float(epe.mean()), float(epe.max()))


@needs_raft
def test_raft_flows_vs_oracle(capi):
    check_raft_flows()


def check_image_propagation(runtime=None):
    """P5: exact mask agreement and fp16-level frame agreement with the oracle."""
    import sys

    from conftest import GOLDEN
    from oracle import propainter_oracle as P

    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from make_golden_propainter import inputs
    from vsr_b200.flow_propagation import _PropRuntime, propagate_images_host

    z = np.load(os.path.join(GOLDEN, "propainter_real.npz"))
    frames, mask = inputs()[:2]
    _, md = P.read_mask(mask, len(frames))
    ff, fb = z["pred_flows_f"][0].astype(np.float32), z["pred_flows_b"][0].astype(np.float32)
    rt = runtime if runtime is not None else _PropRuntime("cuda:0")
    upd, um = propagate_images_host(rt, frames, md[0], ff, fb)
    rt.close()
    x = torch.from_numpy(np.stack([f[:, :, ::-1] for f in frames]).astype(np.float32) / 255).permute(0, 3, 1, 2)[None] * 2 - 1
    masks = torch.from_numpy(np.stack(md).astype(np.float32) / 255)[None, :, None]
    prop, want_m = P.img_propagation(x * (1 - masks), torch.from_numpy(ff)[None], torch.from_numpy(fb)[None], masks)
    want = P.updated_frames(x, masks, prop)[0].numpy()
    assert (um != want_m[0].numpy()).mean() < 1e-4 and np.abs(upd - want).max() < 2e-3


def test_image_propagation_vs_oracle(capi):
    """P5 on the device: needs no checkpoint (the flows are the reference's, stored in tests/golden/propainter_real.npz)."""
    check_image_propagation()


def check_flow_completion(runtime=None):
    """P4.  fp16 simulation: 2.4e-3 px; bar: completed flows within 0.03 px of the oracle."""
    import sys

    from conftest import GOLDEN
    from oracle import propainter_oracle as P
    from oracle import rfc_oracle as C

    path = os.path.join(ROOT, "weights", "propainter", "recurrent_flow_completion.pth")
    if not os.path.exists(path):
        pytest.skip("recurrent_flow_completion.pth not staged")
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from make_golden_propainter import inputs
    from vsr_b200.flow_completion import FlowCompletion

    z = np.load(os.path.join(GOLDEN, "propainter_real.npz"))
    frames, mask = inputs()[:2]
    fm, _ = P.read_mask(mask, len(frames))
    gf, gb = z["gt_flows_f"][0].astype(np.float32), z["gt_flows_b"][0].astype(np.float32)
    pf, pb = FlowCompletion(path, "cuda:0", runtime=runtime).complete_host(gf, gb, fm[0])
    masks = torch.from_numpy(np.stack(fm).astype(np.float32) / 255)[None, :, None]
    wf, wb = C.complete_bidirectional(C.load_weights(path), torch.from_numpy(gf)[None], torch.from_numpy(gb)[None], masks)
    assert np.abs(pf - wf[0].numpy()).max() < 0.03 and np.abs(pb - wb[0].numpy()).max() < 0.03


def test_flow_completion_vs_oracle(capi):
    """P4 on the device (gated)."""
    check_flow_completion()


def test_propainter_pipeline_vs_reference_frames(capi):
    """The whole device pipeline (gated) against the frames of the unmodified reference.  fp16 simulation: 58.9 dB in the hole; bar: PSNR >= 45 dB
    against the reference's `comp` inside the hole; outside the dilated mask bit-exact (the reference copies the input there)."""
    import sys

    from conftest import GOLDEN

    d = os.path.join(ROOT, "weights", "propainter")
    if not all(os.path.exists(os.path.join(d, f)) for f in ("ProPainter.pth", "recurrent_flow_completion.pth", "raft-things.pth")):
        pytest.skip("ProPainter weights not staged")
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from make_golden_propainter import inputs
    from oracle import propainter_oracle as P
    from vsr_b200.propainter_inpaint import PropainterInpaint

    z = np.load(os.path.join(GOLDEN, "propainter_real.npz"))
    frames, mask = inputs()[:2]
    out = np.stack(PropainterInpaint("cuda:0", d).inpaint(frames, mask))
    _, md = P.read_mask(mask, len(frames))
    keep = np.stack(md) == 0
    assert np.array_equal(out[keep], np.stack(frames)[keep])
    hole = ~keep
    assert O.psnr_u8(out[hole].astype(np.float32), z["comp"][hole].astype(np.float32)) >= 45.0


def test_batched_detection_equals_single_frames(capi):
    """`TextDetector.probability_maps` (several sampled frames per launch), gated on the detector model; bar: every frame's map equals its single-frame map to fp16 noise (the scales may differ between the two programs)."""
    import cv2

    model = os.path.join(ROOT, "weights", "V5", "ch_det")
    if not os.path.exists(os.path.join(model, "inference.pdiparams")):
        pytest.skip("detector model not staged")
    from vsr_b200.dbnet import TextDetector

    rng = np.random.default_rng(9)
    imgs = []
    for i in range(4):
        img = cv2.GaussianBlur(rng.integers(0, 255, (360, 640, 3), dtype=np.uint8), (0, 0), 9)
        cv2.putText(img, f"frame {i} text", (80 + 20 * i, 320), cv2.FONT_HERSHEY_SIMPLEX, 1.2, (255, 255, 255), 3, cv2.LINE_AA)
        imgs.append(img)
    det = TextDetector(model, "cuda:0")
    maps = det.probability_maps(imgs)
    for m, img in zip(maps, imgs):
        d = np.abs(m - det.probability_map(img))
        assert d.mean() <= 5e-4 and (d > 0.05).mean() <= 2e-3
