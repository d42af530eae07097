"""The SuperPoint oracle (oracle/superpoint_oracle.py, groundwork for SURVEY.md 8f1) against fixtures produced by the
reference's own superpoint.py (oracle/make_golden_superpoint.py): identical keypoints (integer pixel positions, same
order), scores within 1e-6, descriptors within 1e-5.  CPU only.  The oracle computes in float64 and its keypoints and
scores are compared with the reference's float64 run (tests/golden/float64/): in float32 the convolutions' summation
order, which changes with the host CPU and thread count, moves scores by ~2e-6.  Descriptors are compared with the
float32 run, whose rounding (~4e-7) lies far inside their tolerance."""
import os

import pytest
import torch

from lightglue_b200 import synth
from oracle import superpoint_oracle as sp
from oracle import superpoint_synth as sps

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = sorted(f[:-3] for f in os.listdir(GOLDEN) if f.startswith("sp_") and f.endswith(".pt"))


@pytest.mark.parametrize("name", CASES)
def test_superpoint_oracle_matches_reference_fixture(name):
    fix = torch.load(os.path.join(GOLDEN, name + ".pt"), weights_only=False)
    rc = fix["recipe"]
    w = sps.make_superpoint_state_dict(0)
    for k, v in fix["weights_checksum"].items():
        assert synth.checksum(w[k]) == v, k
    image = sps.make_image(rc["h"], rc["w"], rc["b"], rc["seed"])
    assert synth.checksum(image) == fix["image_checksum"]
    with torch.no_grad():
        out = sp.forward({k: v.double() for k, v in w.items()}, image.double(), **fix["conf"])
    gold = fix["out"]
    gold64 = torch.load(os.path.join(GOLDEN, "float64", name + ".pt"), weights_only=False)
    assert len(out["keypoints"]) == rc["b"]
    for b in range(rc["b"]):
        assert torch.equal(out["keypoints"][b], gold64["keypoints"][b]), "keypoint set / order differs"
        assert float((out["keypoint_scores"][b] - gold64["keypoint_scores"][b]).abs().max()) <= 1e-6
        d = out["descriptors"][b][:: gold["desc_stride"][b]]
        assert d.shape == gold["descriptors"][b].shape
        assert float((d - gold["descriptors"][b]).abs().max()) <= 1e-5
        assert float((out["descriptors"][b].norm(dim=-1) - 1).abs().max()) <= 1e-5
        k = out["keypoints"][b]
        pad = fix["conf"]["remove_borders"]
        assert int(k[:, 0].min()) >= pad and int(k[:, 0].max()) < rc["w"] - pad
        assert int(k[:, 1].min()) >= pad and int(k[:, 1].max()) < rc["h"] - pad


def test_nms_leaves_no_two_keypoints_within_the_radius():
    w = sps.make_superpoint_state_dict(0)
    with torch.no_grad():
        out = sp.forward(w, sps.make_image(160, 240, 1, 21), nms_radius=4)
    k = out["keypoints"][0]
    d = (k[:, None] - k[None]).abs().amax(-1)  # Chebyshev distance = the square NMS window
    d.fill_diagonal_(99)
    assert int(d.min()) > 4
