"""What the reference does with adaptive depth on a batch of more than one pair -- the UNMODIFIED reference file run on the
CPU by oracle/make_golden.py, its outputs stored in tests/golden/batch_early_exit.pt -- and therefore why lightglue_b200
decides per pair (documented deviation, LightGlue.forward docstring, INTEGRATION.md).

lightglue.py:645-656 (`check_if_stop`): the low-confidence count is summed over the WHOLE batch and divided by ONE pair's
m + n, and one decision is taken for all pairs.  So a pair's result depends on its batch-mates -- even on being duplicated:
two copies of a pair that stops early alone run all nine layers together, with different matches.  (With point pruning on,
`torch.where(mask)[1]` at 554 / 562 additionally concatenates the kept columns of all rows: not defined for B > 1.)"""
import os

import pytest
import torch

from lightglue_b200 import synth
from oracle import lightglue_oracle as oracle
from tests.helpers import GOLDEN, compare_outputs


@pytest.fixture(scope="module")
def fixture():
    """The stored reference outputs, and the regenerated weights / pairs they were computed from."""
    fix = torch.load(os.path.join(GOLDEN, "batch_early_exit.pt"), weights_only=False)
    rc = fix["recipe"]
    sd = synth.make_state_dict(adaptive=True, seed=rc["weight_seed"])
    for k, v in fix["weights_checksum"].items():
        assert synth.checksum(sd[k]) == v, f"regenerated weight {k} differs from the fixture's"
    pairs = {}
    for s in rc["seeds"]:
        p = synth.make_pair(rc["n"], b=1, seed=s)[0]
        assert synth.checksum(p["image0"]["keypoints"]) == fix["inputs_checksum"][s]["k0"]
        assert synth.checksum(p["image1"]["descriptors"]) == fix["inputs_checksum"][s]["d1"]
        pairs[s] = p
    return fix, sd, pairs


def test_reference_batched_early_exit_depends_on_batch_mates(fixture):
    ref = fixture[0]["out"]
    alone41, alone42, twice, mixed = ref["alone41"], ref["alone42"], ref["twice41"], ref["mixed"]
    assert alone41["stop"] < alone42["stop"] == 9  # one pair exits early, the other never
    # the SAME pair, twice in one batch, no longer exits: count summed over the batch / one pair's m + n
    assert twice["stop"] == 9 > alone41["stop"]
    assert not torch.equal(twice["matches0"][0], alone41["matches0"][0])  # and its matches changed with it
    assert torch.equal(twice["matches0"][0], twice["matches0"][1])
    assert mixed["stop"] == 9  # one batch-global decision: pair 41 is dragged along


def test_oracle_matches_the_reference_on_each_pair_alone(fixture):
    """The per-pair semantics lightglue_b200 implements (and the GPU tests pin against the oracle) are the reference's
    own answer for a pair matched alone."""
    torch.set_grad_enabled(False)
    fix, sd, pairs = fixture
    rc = fix["recipe"]
    for s in rc["seeds"]:
        out = oracle.forward(sd, pairs[s], depth_confidence=rc["depth_confidence"], width_confidence=rc["width_confidence"])
        compare_outputs(out, fix["out"][f"alone{s}"], score_tol=2e-5)
