"""Shared helpers for the parity tests: rebuild a golden case's inputs/weights and compare outputs."""
import os

import torch

from lightglue_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# matcher fixtures only (sp_* are the SuperPoint extractor oracle's, tests/test_superpoint_oracle_golden.py; batch_* hold
# the reference's B > 1 semantics, tests/test_reference_batch_semantics.py)
ALL_CASES = sorted(f[:-3] for f in os.listdir(GOLDEN) if f.endswith(".pt") and not f.startswith(("sp_", "batch_")))


def load_case(name):
    """Returns (fixture, data, state_dict); asserts regenerated inputs/weights match the fixture's checksums."""
    fix = torch.load(os.path.join(GOLDEN, name + ".pt"), weights_only=False)
    rc = fix["recipe"]
    data, perm = synth.make_pair(
        rc["n"], d=rc["d"], b=rc["b"], seed=rc["seed"], m=rc.get("m"), scale_ori=rc.get("scale_ori", False)
    )
    if rc.get("drop_size"):
        for k in ("image0", "image1"):
            data[k].pop("image_size")
    sd = synth.make_state_dict(
        seed=0, input_dim=rc["d"], adaptive=rc.get("adaptive", False), add_scale_ori=rc.get("scale_ori", False)
    )
    for k, v in fix["weights_checksum"].items():
        assert synth.checksum(sd[k]) == v, f"regenerated weight {k} differs from the fixture's"
    assert synth.checksum(data["image0"]["keypoints"]) == fix["inputs_checksum"]["k0"]
    assert synth.checksum(data["image1"]["descriptors"]) == fix["inputs_checksum"]["d1"]
    return fix, data, sd


def forward_kwargs(fix):
    rc, conf = fix["recipe"], fix["conf"]
    return dict(
        depth_confidence=conf["depth_confidence"],
        width_confidence=conf["width_confidence"],
        filter_threshold=conf["filter_threshold"],
        pruning_threshold=rc.get("pruning_threshold", -1),
        add_scale_ori=rc.get("scale_ori", False),
    )


def compare_outputs(out, gold, *, score_tol, exact_indices=True, max_flips=0):
    """Compare a matcher output dict against a golden `out` dict.  Returns (n_index_flips, max_abs_dscore)."""
    flips = 0
    for k in ("matches0", "matches1"):
        a = out[k].cpu().to(torch.int64)
        b = gold[k].to(torch.int64)
        assert a.shape == b.shape, (k, a.shape, b.shape)
        flips += int((a != b).sum())
    dmax = 0.0
    for k in ("matching_scores0", "matching_scores1"):
        a = out[k].cpu().float()
        b = gold[k].float()
        assert a.shape == b.shape
        if a.numel():
            dmax = max(dmax, float((a - b).abs().max()))
    if exact_indices:
        assert flips <= max_flips, f"{flips} match-index flips (allowed {max_flips})"
    assert dmax <= score_tol, f"max |dscore| {dmax} > {score_tol}"
    assert int(out["stop"]) == int(gold["stop"]), (out["stop"], gold["stop"])
    return flips, dmax
